"""GPU parity: every tf_ops entry point, called through the Python op surface -> ctypes ->
C ABI -> sm_100a kernels, against the CPU oracle (bit-exact for indices and copies, 1e-5 abs
for interpolation) and against what the reference's own CUDA kernels returned on the same inputs
(tests/golden/reference_kernels.*, written by tests/golden/make_reference_golden.py from the
functions named *_reference_inputs / *_REFERENCE_CASES below)."""
import numpy as np
import pytest

from _util import assert_reference, assert_reference_close, golden, golden_inputs, rng_cloud, to_cuda

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops(cuda):
    import pn2_b200  # noqa: F401
    from pn2_b200.tf_ops import tf_grouping, tf_interpolate, tf_sampling
    from oracle import oracle as orc
    return tf_sampling, tf_grouping, tf_interpolate, orc


FPS_CASES = [(2, 1024, 256), (3, 64, 16), (2, 100, 100), (1, 8192, 1024), (2, 5000, 300),
             (4, 256, 64), (1, 513, 40), (2, 2048, 128), (1, 12000, 64), (1, 20000, 32),
             (2, 16, 20)]


@pytest.mark.parametrize("b,n,m", FPS_CASES)
def test_fps_matches_oracle(ops, b, n, m):
    ts, _, _, orc = ops
    x = rng_cloud(100 + n, b, n)
    got = ts.farthest_point_sample(m, to_cuda(x)).cpu().numpy()
    exp = orc.farthest_point_sample(m, x)
    assert got.dtype == np.int32 and got.shape == (b, m)
    np.testing.assert_array_equal(got, exp)


@pytest.mark.parametrize("n,m", [(1500, 200), (700, 64), (4096, 128), (9000, 50)])
def test_fps_tie_order(ops, n, m):
    """Integer-grid clouds: many exactly equal distances and duplicate points.  The winner must
    be the lowest (k mod 512) then lowest k, as the reference's strided scan + tree gives."""
    ts, _, _, orc = ops
    rs = np.random.RandomState(7)
    x = rs.randint(0, 4, (2, n, 3)).astype(np.float32)
    got = ts.farthest_point_sample(m, to_cuda(x)).cpu().numpy()
    np.testing.assert_array_equal(got, orc.farthest_point_sample(m, x))


def test_fps_properties_full_size(ops):
    """Config-2 size: first index 0, all indices distinct and in range, min pairwise distance of
    the prefix is non-increasing (the defining property of farthest point sampling)."""
    ts, _, _, _ = ops
    import torch
    x = rng_cloud(100, 16, 8192, scale=(10, 10, 5), shift=(-5, -5, 0))
    idx = ts.farthest_point_sample(1024, to_cuda(x)).cpu().numpy()
    assert (idx[:, 0] == 0).all() and idx.min() >= 0 and idx.max() < 8192
    for b in range(16):
        assert len(set(idx[b].tolist())) == 1024
    p = torch.as_tensor(x[0][idx[0]], dtype=torch.float64)
    d = torch.cdist(p, p)
    sel = []
    for j in range(1, 64):
        sel.append(d[j, :j].min().item())
    assert all(sel[i] >= sel[i + 1] - 1e-9 for i in range(len(sel) - 1))


def fps_reference_inputs():
    """(key, cloud, npoint) of the FPS comparisons with the reference's kernel."""
    for b, n, m in [(2, 1024, 256), (16, 8192, 1024), (3, 5000, 333)]:
        yield "fps_%d_%d_%d" % (b, n, m), rng_cloud(5 + n, b, n), m
    yield "fps_lattice_2_3000_400", np.random.RandomState(3).randint(0, 5, (2, 3000, 3)).astype(np.float32), 400


def test_fps_matches_reference_kernel(ops):
    ts, _, _, _ = ops
    for key, x, m in fps_reference_inputs():
        assert_reference(key, ts.farthest_point_sample(m, to_cuda(x)))


def test_gather_point_and_grad(ops):
    ts, _, _, orc = ops
    import torch
    x = rng_cloud(1, 3, 777)
    idx = np.random.RandomState(2).randint(0, 777, (3, 200)).astype(np.int32)
    xt = to_cuda(x).requires_grad_(True)
    out = ts.gather_point(xt, to_cuda(idx))
    np.testing.assert_array_equal(out.detach().cpu().numpy(), orc.gather_point(x, idx))
    g = np.random.RandomState(3).random_sample((3, 200, 3)).astype(np.float32)
    out.backward(to_cuda(g))
    np.testing.assert_allclose(xt.grad.cpu().numpy(), orc.gather_point_grad(x.shape, idx, g),
                               atol=1e-5)
    np.testing.assert_allclose(ts.gather_point_grad(xt.detach(), to_cuda(idx), to_cuda(g)).cpu().numpy(),
                               orc.gather_point_grad(x.shape, idx, g), atol=1e-5)


BALL_CASES = [  # b, n, m, radius, nsample
    (2, 1024, 256, 0.2, 32),     # config 1: truncation and padding both occur
    (16, 8192, 1024, 0.5, 32),   # SA1 of config 2 on the unit cube: truncation everywhere
    (2, 333, 77, 0.15, 16),      # ragged n (no TMA path), small
    (1, 4096, 4096, 0.05, 64),   # many queries -> streaming kernel
    (3, 64, 16, 0.4, 32),        # tiny
    (2, 1000, 10, 0.01, 8),      # almost no hits: zero rows
    (1, 2050, 130, 0.3, 128),    # nsample 128, n % 4 != 0
    (40, 2048, 512, 0.12, 24),   # enough queries for SPLIT=1 with several tiles
]


@pytest.mark.parametrize("b,n,m,radius,ns", BALL_CASES)
def test_query_ball_point_matches_oracle(ops, b, n, m, radius, ns):
    _, tg, _, orc = ops
    x1 = rng_cloud(11 + n, b, n)
    x2 = x1[:, :m].copy() if m <= n else rng_cloud(12, b, m)
    if b == 2 and n == 1000:
        x2 = rng_cloud(99, b, m)  # unrelated queries: rows with no hit at all
    idx, cnt = tg.query_ball_point(radius, ns, to_cuda(x1), to_cuda(x2))
    eidx, ecnt = orc.query_ball_point(radius, ns, x1, x2)
    np.testing.assert_array_equal(cnt.cpu().numpy(), ecnt)
    np.testing.assert_array_equal(idx.cpu().numpy(), eidx)


def test_query_ball_boundary_radius(ops):
    """Points at distances straddling the radius by single ulps: the d2 < T rewrite must agree
    with the reference predicate max(sqrtf(d2),1e-20f) < radius everywhere."""
    _, tg, _, orc = ops
    rs = np.random.RandomState(5)
    for radius in [0.1, 0.5, 1.0, 0.3333333, 2.0, 4.0, 1e-3]:
        q = np.zeros((1, 1, 3), np.float32)
        r32 = np.float32(radius)
        # distances around the radius along x, every ulp in +-40
        xs = [r32]
        for _ in range(40):
            xs.append(np.nextafter(xs[-1], np.float32(np.inf)))
        lo = r32
        for _ in range(40):
            lo = np.nextafter(lo, np.float32(0))
            xs.append(lo)
        pts = np.zeros((1, len(xs) + 200, 3), np.float32)
        pts[0, :len(xs), 0] = np.array(xs, np.float32)
        rnd = rs.normal(size=(200, 3))
        rnd = rnd / np.linalg.norm(rnd, axis=1, keepdims=True) * radius * (1 + rs.uniform(-1e-6, 1e-6, (200, 1)))
        pts[0, len(xs):] = rnd.astype(np.float32)
        ns = pts.shape[1]
        idx, cnt = tg.query_ball_point(float(radius), ns, to_cuda(pts), to_cuda(q))
        eidx, ecnt = orc.query_ball_point(float(radius), ns, pts, q)
        np.testing.assert_array_equal(cnt.cpu().numpy(), ecnt)
        np.testing.assert_array_equal(idx.cpu().numpy(), eidx)


def ball_reference_inputs():
    """(key, radius, nsample, cloud, queries) of the ball-query comparisons with the reference's kernel."""
    for b, n, m, radius, ns in [(2, 1024, 256, 0.2, 32), (16, 8192, 1024, 0.1, 32),
                                (4, 2048, 512, 0.25, 64)]:
        x1 = rng_cloud(21 + n, b, n)
        yield "ball_%d_%d_%d_%g_%d" % (b, n, m, radius, ns), radius, ns, x1, np.ascontiguousarray(x1[:, :m])


def test_query_ball_matches_reference_kernel(ops):
    _, tg, _, _ = ops
    for key, radius, ns, x1, x2 in ball_reference_inputs():
        idx, cnt = tg.query_ball_point(radius, ns, to_cuda(x1), to_cuda(x2))
        assert_reference(key + "_cnt", cnt)
        assert_reference(key + "_idx", idx)


def test_query_ball_validation(ops):
    _, tg, _, _ = ops
    x = to_cuda(rng_cloud(1, 1, 32))
    with pytest.raises(ValueError, match="positive radius"):
        tg.query_ball_point(0.0, 8, x, x)
    with pytest.raises(ValueError, match="positive nsample"):
        tg.query_ball_point(0.1, 0, x, x)
    with pytest.raises(ValueError, match="xyz1 shape"):
        tg.query_ball_point(0.1, 8, x[..., :2], x)


@pytest.mark.parametrize("c", [3, 16, 64, 67, 128])
def test_group_point_and_grad(ops, c):
    _, tg, _, orc = ops
    rs = np.random.RandomState(c)
    pts = rs.random_sample((2, 300, c)).astype(np.float32)
    idx = rs.randint(0, 300, (2, 40, 8)).astype(np.int32)
    pt = to_cuda(pts).requires_grad_(True)
    out = tg.group_point(pt, to_cuda(idx))
    np.testing.assert_array_equal(out.detach().cpu().numpy(), orc.group_point(pts, idx))
    g = rs.random_sample((2, 40, 8, c)).astype(np.float32)
    out.backward(to_cuda(g))
    np.testing.assert_allclose(pt.grad.cpu().numpy(), orc.group_point_grad(pts.shape, idx, g),
                               atol=1e-5)


def test_group_point_grad_check_like_reference(ops):
    """tf_ops/test_tf_ops.py:38-56: finite-difference gradient error of group_point(points,
    query_ball_point(0.3, 32, xyz1, xyz2)) w.r.t. points (1,128,16) below 1e-4.  group_point is
    linear in points, so the analytic vector-Jacobian product must equal the directional
    finite difference up to fp32 rounding."""
    import torch
    _, tg, _, _ = ops
    rs = np.random.RandomState(0)
    points = to_cuda(rs.random_sample((1, 128, 16)).astype(np.float32))
    xyz1 = to_cuda(rs.random_sample((1, 128, 3)).astype(np.float32))
    xyz2 = to_cuda(rs.random_sample((1, 8, 3)).astype(np.float32))
    idx, _ = tg.query_ball_point(0.3, 32, xyz1, xyz2)
    p = points.clone().requires_grad_(True)
    out = tg.group_point(p, idx)
    v = to_cuda(rs.random_sample(tuple(out.shape)).astype(np.float32))
    out.backward(v)
    for _ in range(4):
        d = to_cuda(rs.normal(size=(1, 128, 16)).astype(np.float32))
        fd = ((tg.group_point(points + 1e-2 * d, idx) - tg.group_point(points - 1e-2 * d, idx))
              / 2e-2 * v).sum().item()
        an = (p.grad * d).sum().item()
        assert abs(fd - an) / max(1.0, abs(an)) < 1e-4


def test_three_nn_golden_vector(ops):
    """The reference's only known-answer test, tf_ops/test_interpolate.py:6-35 (seed 100,
    (64,8192,3) targets, (64,1024,3) references)."""
    _, _, ti, _ = ops
    np.random.seed(100)
    target = np.random.random((64, 8192, 3)).astype("float32")
    reference = np.random.random((64, 1024, 3)).astype("float32")
    dist, idx = ti.three_nn(to_cuda(target), to_cuda(reference))
    dist, idx = dist.cpu().numpy(), idx.cpu().numpy()
    assert dist.shape == (64, 8192, 3) and idx.dtype == np.int32 and dist.dtype == np.float32
    exp_d = np.array([0.00175864, 0.00671887, 0.0034472, 0.00337327, 0.00191902, 0.00075543,
                      0.00169418, 0.00473733, 0.00381071], np.float32)
    exp_i = np.array([137, 856, 116, 76, 915, 199, 117, 659, 786])
    np.testing.assert_allclose(dist[:3, :3, :1].flatten(), exp_d, atol=5e-9)
    np.testing.assert_array_equal(idx[:3, :3, :1].flatten(), exp_i)


@pytest.mark.parametrize("b,n,m", [(2, 512, 128), (1, 1000, 3), (3, 77, 1500), (16, 8192, 1024)])
def test_three_nn_matches_oracle(ops, b, n, m):
    _, _, ti, orc = ops
    x1, x2 = rng_cloud(31 + n, b, n), rng_cloud(32 + m, b, m)
    dist, idx = ti.three_nn(to_cuda(x1), to_cuda(x2))
    ed, ei = orc.three_nn(x1, x2, threads=8)
    np.testing.assert_array_equal(idx.cpu().numpy(), ei)
    np.testing.assert_array_equal(dist.cpu().numpy(), ed)  # same fp64 ops, same cast: bit-exact


def test_three_nn_ties_lowest_index(ops):
    _, _, ti, orc = ops
    rs = np.random.RandomState(4)
    x2 = rs.randint(0, 3, (2, 200, 3)).astype(np.float32)
    x1 = rs.randint(0, 3, (2, 50, 3)).astype(np.float32)
    dist, idx = ti.three_nn(to_cuda(x1), to_cuda(x2))
    ed, ei = orc.three_nn(x1, x2)
    np.testing.assert_array_equal(idx.cpu().numpy(), ei)
    np.testing.assert_array_equal(dist.cpu().numpy(), ed)


@pytest.mark.parametrize("c", [16, 64, 131, 512])
def test_three_interpolate_and_grad(ops, c):
    """Forward within 1e-5 abs of the oracle (in fact bit-exact: same mul/add sequence);
    gradient against the oracle's scatter (atomics reorder the sums: 1e-5 abs)."""
    _, _, ti, orc = ops
    rs = np.random.RandomState(c)
    pts = rs.random_sample((2, 128, c)).astype(np.float32)
    x1, x2 = rng_cloud(41, 2, 512), rng_cloud(42, 2, 128)
    dist, idx = ti.three_nn(to_cuda(x1), to_cuda(x2))
    w = rs.random_sample((2, 512, 3)).astype(np.float32)
    w /= w.sum(-1, keepdims=True)
    pt = to_cuda(pts).requires_grad_(True)
    out = ti.three_interpolate(pt, idx, to_cuda(w))
    exp = orc.three_interpolate(pts, idx.cpu().numpy(), w)
    np.testing.assert_allclose(out.detach().cpu().numpy(), exp, atol=1e-5)
    np.testing.assert_array_equal(out.detach().cpu().numpy(), exp)
    g = rs.random_sample((2, 512, c)).astype(np.float32)
    out.backward(to_cuda(g))
    eg = orc.three_interpolate_grad(pts.shape, idx.cpu().numpy(), w, g)
    np.testing.assert_allclose(pt.grad.cpu().numpy(), eg, atol=1e-5, rtol=1e-5)


def test_three_interpolate_grad_check_like_reference(ops):
    """tf_ops/test_tf_ops.py:80-94: weights 1/3, points (1,8,16) -> (1,128,16), error < 1e-4."""
    _, _, ti, _ = ops
    rs = np.random.RandomState(0)
    points = to_cuda(rs.random_sample((1, 8, 16)).astype(np.float32))
    xyz1 = to_cuda(rs.random_sample((1, 128, 3)).astype(np.float32))
    xyz2 = to_cuda(rs.random_sample((1, 8, 3)).astype(np.float32))
    dist, idx = ti.three_nn(xyz1, xyz2)
    import torch
    weight = torch.ones_like(dist) / 3.0
    p = points.clone().requires_grad_(True)
    out = ti.three_interpolate(p, idx, weight)
    v = to_cuda(rs.random_sample(tuple(out.shape)).astype(np.float32))
    out.backward(v)
    for _ in range(4):
        d = to_cuda(rs.normal(size=(1, 8, 16)).astype(np.float32))
        fd = ((ti.three_interpolate(points + 1e-2 * d, idx, weight)
               - ti.three_interpolate(points - 1e-2 * d, idx, weight)) / 2e-2 * v).sum().item()
        an = (p.grad * d).sum().item()
        assert abs(fd - an) / max(1.0, abs(an)) < 1e-4


def _selection_cases():
    rs = np.random.RandomState(9)
    nan = rs.randint(0, 4, (1, 12, 150)).astype(np.float32)
    nan[0, :, ::7] = np.nan
    nan[0, 3, 0] = np.nan
    inf = rs.randint(0, 3, (1, 9, 100)).astype(np.float32)
    inf[inf == 2] = np.inf
    return {"random": rs.random_sample((2, 20, 300)), "ties4": rs.randint(0, 4, (2, 33, 257)),
            "ties2": rs.randint(0, 2, (1, 17, 64)), "zeros": np.zeros((1, 5, 90)), "nan": nan, "inf": inf,
            "wide": rs.random_sample((1, 3, 5000)), "narrow": rs.randint(0, 3, (2, 7, 9))}


@pytest.mark.parametrize("name", sorted(_selection_cases()))
@pytest.mark.parametrize("k", [1, 16, 128])
def test_select_top_k_matches_oracle_and_reference_kernel(ops, name, k):
    """The WHOLE output rows (first k and the permuted tail) against the C oracle and against the
    reference's own selection_sort_gpu -- ties, NaN and inf included."""
    _, tg, _, orc = ops
    d = np.ascontiguousarray(_selection_cases()[name], np.float32)
    if k > d.shape[2] and d.shape[2] > 128:
        pytest.skip("k > 128 with n > 128 is not supported")
    dd = to_cuda(d)
    outi, out = tg.select_top_k(k, dd)
    ei, eo = orc.select_top_k(k, d)
    np.testing.assert_array_equal(outi.cpu().numpy(), ei)
    np.testing.assert_array_equal(out.cpu().numpy().view(np.uint32), eo.view(np.uint32))
    assert_reference("select_%s_k%d_idx" % (name, k), outi)
    assert_reference("select_%s_k%d_val" % (name, k), out)


def _sqdist_matrix(x1, x2):
    """(b,m,n) fp32 matrix exactly as tf_grouping.py:79-82 evaluates it (left to right, no fma)."""
    d = (x1[:, None, :, :] - x2[:, :, None, :]).astype(np.float32)
    sq = (d * d).astype(np.float32)
    acc = sq[..., 0]
    for a in range(1, sq.shape[-1]):
        acc = (acc + sq[..., a]).astype(np.float32)
    return acc


KNN_REFERENCE_CASES = [(2, 1024, 256, 32, 3, "uniform"), (32, 512, 128, 32, 3, "uniform"),
                       (1, 8192, 100, 64, 3, "uniform"), (2, 300, 50, 16, 3, "lattice"),
                       (1, 200, 30, 128, 3, "duplicates"), (2, 400, 60, 8, 5, "uniform"),
                       (1, 64, 10, 64, 2, "lattice")]


def knn_reference_inputs(b, n, m, k, c, kind):
    """(key, x1, x2) of a knn_point case; the reference's selection kernel ran on _sqdist_matrix(x1, x2)."""
    rs = np.random.RandomState(n + k)
    if kind == "uniform":
        x1, x2 = rs.random_sample((b, n, c)), rs.random_sample((b, m, c))
    elif kind == "lattice":
        x1, x2 = rs.randint(0, 4, (b, n, c)), rs.randint(0, 4, (b, m, c))
    else:
        x1 = np.repeat(rs.random_sample((b, n // 4, c)), 4, 1)
        x2 = x1[:, :m] + 0.0
    key = "knn_%d_%d_%d_%d_%d_%s" % (b, n, m, k, c, kind)
    return key, np.ascontiguousarray(x1, np.float32), np.ascontiguousarray(x2, np.float32)


@pytest.mark.parametrize("b,n,m,k,c,kind", KNN_REFERENCE_CASES)
def test_knn_point_fused_matches_oracle_and_reference_selection(ops, b, n, m, k, c, kind):
    """knn_point (one fused kernel, no (b,m,n) tensor) == the oracle restatement of tf_grouping.py:64-89 ==
    the reference's own selection kernel applied to the fp32 distance matrix; (32,512)/(32,128), k=32 is the
    reference's smoke-test shape (test_tf_ops.py:9-24)."""
    _, tg, _, orc = ops
    key, x1, x2 = knn_reference_inputs(b, n, m, k, c, kind)
    val, idx = tg.knn_point(k, to_cuda(x1), to_cuda(x2))
    ev, ei = orc.knn_point(k, x1, x2)
    np.testing.assert_array_equal(idx.cpu().numpy(), ei)
    np.testing.assert_array_equal(val.cpu().numpy().view(np.uint32), ev.view(np.uint32))
    assert_reference(key + "_idx", idx)  # the first k columns of the reference's selection
    assert_reference(key + "_val", val)


def test_knn_point_validation(ops):
    _, tg, _, _ = ops
    x = to_cuda(rng_cloud(1, 1, 50))
    with pytest.raises(ValueError, match="positive k"):
        tg.knn_point(0, x, x)
    with pytest.raises(ValueError, match="must not exceed"):
        tg.knn_point(51, x, x)


def gather_group_reference_inputs():
    """(cloud, gradient of the 256 gathered points, [(c, points, gradient of the grouped points)]); the gathers
    take FPS(256) of the cloud, the groups the ball query (0.2, 32) around those points."""
    rs = np.random.RandomState(4)
    x = rs.random_sample((16, 8192, 3)).astype(np.float32)
    g = rs.normal(size=(16, 256, 3)).astype(np.float32)
    groups = [(c, rs.random_sample((16, 8192, c)).astype(np.float32),
               rs.normal(size=(16, 256, 32, c)).astype(np.float32)) for c in (3, 16, 67)]
    return x, g, groups


def test_gather_and_group_match_reference_kernels(ops):
    """gather_point / group_point and their gradients against the reference's own kernels: exact for the
    gathers and for gather_point's gradient (FPS indices are distinct: one addition per element); group_point's
    gradient adds up to 32 contributions per element with fp32 atomics on both sides: 2e-5."""
    ts, tg, _, _ = ops
    x, g, groups = gather_group_reference_inputs()
    x = to_cuda(x)
    fps = ts.farthest_point_sample(256, x)
    assert_reference("gather_point", ts.gather_point(x, fps))
    assert_reference("gather_point_grad", ts.gather_point_grad(x, fps, to_cuda(g)))
    new = ts.gather_point(x, fps)
    idx, _ = tg.query_ball_point(0.2, 32, x, new)
    for c, pts, go in groups:
        pts = to_cuda(pts)
        assert_reference("group_point_c%d" % c, tg.group_point(pts, idx))
        assert_reference_close("group_point_grad_c%d" % c, tg.group_point_grad(pts, idx, to_cuda(go)),
                               atol=2e-5, rtol=1e-5)


# ---------------------------------------------------------------- prob_sample (SURVEY 8f-1)
PROB_CASES = [(1, 5, 8192), (2, 1, 16), (3, 33, 100), (2, 1024, 1000), (2, 4099, 300),
              (2, 8192, 500), (2, 8193, 500), (1, 20000, 3000), (4, 16389, 64), (40, 257, 33)]


def _prob_inputs(b, n, m):
    rs = np.random.RandomState(100 + n)
    p = (rs.random_sample((b, n)) * rs.choice([1e-3, 1.0, 37.0], size=(b, n))).astype(np.float32)
    p[:, rs.randint(0, n, max(1, n // 7))] = 0  # zero-weight categories: flat CDF steps
    r = rs.random_sample((b, m)).astype(np.float32)
    r[:, 0] = 0.0
    if m > 1:
        r[:, 1] = np.nextafter(np.float32(1), np.float32(0))
    return p, r


@pytest.mark.parametrize("b,n,m", PROB_CASES)
def test_prob_sample_matches_oracle(ops, b, n, m):
    """Indices bit-exact; the CDF itself (pn2_cumsum) bit-exact: the kernel reproduces the
    reference's fp32 addition order (tf_sampling.cu:7-92) with warp shuffles."""
    import torch
    from pn2_b200._ffi import F32, call, ptr
    ts, _, _, orc = ops
    p, r = _prob_inputs(b, n, m)
    got = ts.prob_sample(to_cuda(p), to_cuda(r)).cpu().numpy()
    assert got.dtype == np.int32 and got.shape == (b, m)
    np.testing.assert_array_equal(got, orc.prob_sample(p, r))
    pc = to_cuda(p)
    cdf = torch.empty_like(pc)
    call("pn2_cumsum", b, n, ptr(pc, F32), ptr(cdf, F32))
    np.testing.assert_array_equal(cdf.cpu().numpy().view(np.uint32), orc.cumsum(p).view(np.uint32))


PROB_REFERENCE_CASES = [(1, 5, 8192), (2, 8193, 500), (3, 20000, 2000), (32, 1000, 100)]


def test_prob_sample_matches_reference_kernel(ops):
    """Against the reference's own cumsumKernel + binarysearchKernel: indices and CDF."""
    import torch
    from pn2_b200._ffi import F32, call, ptr
    ts, _, _, _ = ops
    for b, n, m in PROB_REFERENCE_CASES:
        p, r = _prob_inputs(b, n, m)
        pc, rc = to_cuda(p), to_cuda(r)
        got = ts.prob_sample(pc, rc)
        assert_reference("prob_%d_%d_%d_idx" % (b, n, m), got)
        cdf = torch.empty_like(pc)
        call("pn2_cumsum", b, n, ptr(pc, F32), ptr(cdf, F32))
        assert_reference("prob_%d_%d_%d_cdf" % (b, n, m), cdf)


def test_prob_sample_like_reference_test(ops):
    """tf_ops/test_tf_ops.py:96-128 (TestSampling): triangle areas -> prob_sample -> gather_point
    -> barycentric points -> farthest_point_sample(1024) -> gather_point, checked op by op."""
    import torch
    ts, _, _, orc = ops
    np.random.seed(100)
    tri = np.random.rand(1, 5, 3, 3).astype("float32")
    a, b, c = (np.ascontiguousarray(tri[:, :, i]) for i in range(3))
    areas = np.sqrt((np.cross(b - a, c - a) ** 2).sum(2) + 1e-9).astype(np.float32)
    r = np.random.rand(1, 8192).astype(np.float32)
    ids = ts.prob_sample(to_cuda(areas), to_cuda(r))
    np.testing.assert_array_equal(ids.cpu().numpy(), orc.prob_sample(areas, r))
    us, vs = (torch.as_tensor(np.random.rand(1, 8192).astype(np.float32)).cuda() for _ in range(2))
    upv, umv = 1 - (us + vs - 1).abs(), us - vs
    us, vs = (upv + umv) * 0.5, (upv - umv) * 0.5
    ta, tb, tc = (ts.gather_point(to_cuda(t), ids) for t in (a, b, c))
    np.testing.assert_array_equal(ta.cpu().numpy(), orc.gather_point(a, ids.cpu().numpy()))
    pts = (ta + (tb - ta) * us[..., None] + (tc - ta) * vs[..., None]).contiguous()
    fps = ts.farthest_point_sample(1024, pts)
    np.testing.assert_array_equal(fps.cpu().numpy(),
                                  orc.farthest_point_sample(1024, pts.cpu().numpy()))
    red = ts.gather_point(pts, fps)
    assert red.shape == (1, 1024, 3) and bool(torch.isfinite(red).all())


def test_prob_sample_validation(ops):
    import torch
    ts, _, _, _ = ops
    p = torch.ones((2, 5), device="cuda")
    with pytest.raises(ValueError, match="num_choices"):
        ts.prob_sample(torch.ones((2, 5, 1), device="cuda"), torch.ones((2, 3), device="cuda"))
    with pytest.raises(ValueError, match="num_points"):
        ts.prob_sample(p, torch.ones((3, 3), device="cuda"))
    assert ts.prob_sample(p, torch.zeros((2, 0), device="cuda")).shape == (2, 0)


# ------------------------------------------- interpolate_label_with_color (SURVEY 8f-3)
def _vote_inputs(seed, ns, nd, nlabels=9, grid=False):
    rs = np.random.RandomState(seed)
    if grid:  # integer lattice: many exactly equal distances and duplicate points
        sp = rs.randint(0, 5, (ns, 3)).astype(np.float32)
        dp = rs.randint(0, 5, (nd, 3)).astype(np.float32)
    else:
        sp = rs.random_sample((ns, 3)).astype(np.float32)
        dp = rs.random_sample((nd, 3)).astype(np.float32)
    sl = rs.randint(0, nlabels, (ns,)).astype(np.int32)
    return sp, sl, dp


@pytest.mark.parametrize("ns,nd,knn", [(500, 3000, 3), (1024, 777, 1), (1025, 1000, 5), (3000, 2049, 4),
                                       (5000, 513, 8), (2500, 300, 9), (2100, 256, 16), (1500, 200, 17),
                                       (1200, 100, 32), (2, 100, 3), (1, 10, 3)])
def test_interpolate_label_with_color_matches_oracle(ops, ns, nd, knn):
    _, _, ti, orc = ops
    sp, sl, dp = _vote_inputs(ns + knn, ns, nd)
    lab, col = ti.interpolate_label_with_color(to_cuda(sp), to_cuda(sl), to_cuda(dp), knn)
    assert lab.dtype.is_floating_point is False and tuple(lab.shape) == (nd,)
    assert str(col.dtype) == "torch.uint8" and tuple(col.shape) == (nd, 3)
    elab, ecol = orc.interpolate_label_with_color(sp, sl, dp, knn)
    np.testing.assert_array_equal(lab.cpu().numpy(), elab)
    np.testing.assert_array_equal(col.cpu().numpy(), ecol)


@pytest.mark.parametrize("knn", [1, 3, 6])
def test_interpolate_label_ties_lowest_index(ops, knn):
    """Equal distances resolve to the lowest sparse index, and the vote keeps the label that first
    reaches the top count in nearest-first order (tf_interpolate.cpp:97-106)."""
    _, _, ti, orc = ops
    sp, sl, dp = _vote_inputs(11, 900, 700, nlabels=4, grid=True)
    lab, col = ti.interpolate_label_with_color(to_cuda(sp), to_cuda(sl), to_cuda(dp), knn)
    elab, ecol = orc.interpolate_label_with_color(sp, sl, dp, knn)
    np.testing.assert_array_equal(lab.cpu().numpy(), elab)
    np.testing.assert_array_equal(col.cpu().numpy(), ecol)


def test_interpolate_label_knn1_is_nearest_label_and_color_table(ops):
    """knn=1 must return the label of the nearest sparse point (checked with three_nn) and the
    colours of tf_interpolate.cpp:46-48; labels outside the table get (0,0,0)."""
    import torch
    _, _, ti, _ = ops
    sp, sl, dp = _vote_inputs(5, 4000, 6000, nlabels=11)
    lab, col = ti.interpolate_label_with_color(to_cuda(sp), to_cuda(sl), to_cuda(dp), 1)
    _, i3 = ti.three_nn(to_cuda(dp[None]), to_cuda(sp[None]))
    np.testing.assert_array_equal(lab.cpu().numpy(), sl[i3[0, :, 0].cpu().numpy()])
    table = np.array([[255, 255, 255], [0, 0, 255], [128, 0, 0], [255, 0, 255], [0, 128, 0],
                      [255, 0, 0], [128, 0, 128], [0, 0, 128], [128, 128, 0], [0, 0, 0], [0, 0, 0]],
                     np.uint8)
    np.testing.assert_array_equal(col.cpu().numpy(), table[lab.cpu().numpy()])


def test_interpolate_label_validation(ops):
    import torch
    _, _, ti, _ = ops
    sp = torch.zeros((4, 3), device="cuda")
    sl = torch.zeros((4,), dtype=torch.int32, device="cuda")
    dp = torch.zeros((5, 3), device="cuda")
    with pytest.raises(ValueError, match="sparse_points must be"):
        ti.interpolate_label_with_color(torch.zeros((4, 2), device="cuda"), sl, dp, 3)
    with pytest.raises(ValueError, match="sparse_labels must be"):
        ti.interpolate_label_with_color(sp, sl[:3], dp, 3)
    with pytest.raises(ValueError, match="dense_points must be"):
        ti.interpolate_label_with_color(sp, sl, torch.zeros((5,), device="cuda"), 3)
    with pytest.raises(ValueError, match="knn must be"):
        ti.interpolate_label_with_color(sp, sl, dp, 0)
    lab, col = ti.interpolate_label_with_color(sp, sl, dp[:0], 3)
    assert tuple(lab.shape) == (0,) and tuple(col.shape) == (0, 3)


# ------------------------------------------------ FPS: thread-block-cluster kernel (config 5)
CLUSTER_CASES = [(1, 12000, 64), (1, 20000, 32), (2, 16389, 100), (3, 40000, 150), (1, 65536, 300),
                 (1, 262144, 200), (16, 16384, 64), (2, 100, 120), (5, 9000, 40)]


def _fps_cluster(x, m):
    import torch
    from pn2_b200._ffi import F32, I32, call, ptr
    b, n, _ = x.shape
    out = torch.empty((b, m), dtype=I32, device=x.device)
    call("pn2_fps_cluster", b, n, m, ptr(x, F32), ptr(out, I32))
    return out


@pytest.mark.parametrize("b,n,m", CLUSTER_CASES)
def test_fps_cluster_matches_oracle(ops, b, n, m):
    """One cluster of up to 16 CTAs per cloud, candidates exchanged through distributed shared
    memory: bit-identical indices to the oracle (and therefore to every other FPS kernel)."""
    _, _, _, orc = ops
    x = rng_cloud(300 + n, b, n)
    got = _fps_cluster(to_cuda(x), m).cpu().numpy()
    np.testing.assert_array_equal(got, orc.farthest_point_sample(m, x, threads=8))


def test_fps_cluster_tie_order(ops):
    """Integer lattice (thousands of exactly equal distances, duplicates): the winner must be the
    lowest (k mod 512) then lowest k ACROSS the CTAs of the cluster as well."""
    _, _, _, orc = ops
    rs = np.random.RandomState(9)
    for n, m in [(20000, 300), (33000, 200)]:
        x = rs.randint(0, 6, (2, n, 3)).astype(np.float32)
        got = _fps_cluster(to_cuda(x), m).cpu().numpy()
        np.testing.assert_array_equal(got, orc.farthest_point_sample(m, x, threads=8))


def test_fps_cluster_matches_reference_kernel(ops):
    assert_reference("fps_cluster_2_30000_256", _fps_cluster(to_cuda(rng_cloud(77, 2, 30000)), 256))


# ------------------------------------------------------------- committed golden fixtures
def test_kernels_match_committed_fixtures(ops):
    """tests/golden/*.npz (oracle outputs frozen by make_golden.py on the seed-100 streams; the
    three_nn one starts from the reference's own golden input, test_interpolate.py:7-10): the
    CUDA path must reproduce every file bit for bit."""
    import torch
    from pn2_b200._ffi import F32, call, ptr
    ts, tg, ti, _ = ops
    inp = golden_inputs()
    fx = golden("three_nn_seed100")
    dist, idx = ti.three_nn(to_cuda(inp["nn_q"]), to_cuda(inp["nn_known"]))
    np.testing.assert_array_equal(idx.cpu().numpy(), fx["idx"])
    np.testing.assert_array_equal(dist.cpu().numpy(), fx["dist"])
    fx = golden("fps_ball_seed100")
    x = to_cuda(inp["xyz"])
    fps = ts.farthest_point_sample(256, x)
    np.testing.assert_array_equal(fps.cpu().numpy(), fx["fps"])
    bidx, bcnt = tg.query_ball_point(0.2, 32, x, ts.gather_point(x, fps))
    np.testing.assert_array_equal(bidx.cpu().numpy(), fx["idx"])
    np.testing.assert_array_equal(bcnt.cpu().numpy(), fx["cnt"])
    fx = golden("prob_vote_seed100")
    ids = ts.prob_sample(to_cuda(inp["areas"]), to_cuda(inp["r"]))
    np.testing.assert_array_equal(ids.cpu().numpy(), fx["ids"])
    w = to_cuda(inp["w"])
    cdf = torch.empty_like(w)
    call("pn2_cumsum", 1, w.shape[1], ptr(w, F32), ptr(cdf, F32))
    np.testing.assert_array_equal(cdf.cpu().numpy().view(np.uint32), fx["cdf"].view(np.uint32))
    lab, col = ti.interpolate_label_with_color(to_cuda(inp["sp"]), to_cuda(inp["sl"]),
                                               to_cuda(inp["dp"]), 3)
    np.testing.assert_array_equal(lab.cpu().numpy(), fx["vote_labels"])
    np.testing.assert_array_equal(col.cpu().numpy(), fx["vote_colors"])
