"""GPU: the optimizer step and the training loop around the path (train.py:387-388, 225-244)."""
import numpy as np
import pytest

from _util import to_cuda

pytestmark = pytest.mark.gpu


def adam_reference(p, g, m, v, lr, b1, b2, eps, t, gscale):
    """tf.train.AdamOptimizer in fp64: lr_t = lr*sqrt(1-b2^t)/(1-b1^t), "epsilon hat" added to sqrt(v)."""
    g = g.astype(np.float64) * gscale
    m = m + (g - m) * (1 - b1)
    v = v + (g * g - v) * (1 - b2)
    lr_t = lr * np.sqrt(1 - b2 ** t) / (1 - b1 ** t)
    return p - lr_t * m / (np.sqrt(v) + eps), m, v


@pytest.mark.parametrize("t,gscale", [(1, 1.0), (7, 0.5), (1000, 0.125)])
def test_adam_step_matches_fp64_formula(cuda, t, gscale):
    import pn2_b200  # noqa: F401
    from pn2_b200._ffi import F32, call, ptr
    rs = np.random.RandomState(t)
    n = 100003
    p = rs.normal(size=n).astype(np.float32)
    g = (rs.normal(size=n) * rs.choice([1e-6, 1e-2, 10.0], size=n)).astype(np.float32)
    g[:100] = 0.0  # e.g. the biases in front of a train-mode BatchNorm
    m = (rs.normal(size=n) * 1e-2).astype(np.float32) if t > 1 else np.zeros(n, np.float32)
    v = (rs.random_sample(n) * 1e-3).astype(np.float32) if t > 1 else np.zeros(n, np.float32)
    # the hyper-parameters cross the C ABI as floats: the reference uses the same rounded values
    # (1 - float(0.999) differs from 0.001 by 1.3e-5 relative, far above the comparison tolerance)
    lr, b1, b2, eps = (float(np.float32(x)) for x in (1e-3, 0.9, 0.999, 1e-8))
    ep, em, ev = adam_reference(p.astype(np.float64), g, m.astype(np.float64), v.astype(np.float64),
                                lr, b1, b2, eps, t, gscale)
    dp, dg, dm, dv = to_cuda(p), to_cuda(g), to_cuda(m), to_cuda(v)
    call("pn2_adam_step", n, ptr(dp, F32), ptr(dg, F32), ptr(dm, F32), ptr(dv, F32), 1e-3, 0.9, 0.999, 1e-8,
         t, gscale)
    # fp32 evaluation: relative 2e-6, plus an absolute floor where m + (g-m)*(1-b1) cancels (|m| ~ 1e-2)
    np.testing.assert_allclose(dm.cpu().numpy(), em, rtol=2e-6, atol=1e-8)
    np.testing.assert_allclose(dv.cpu().numpy(), ev, rtol=2e-6, atol=1e-9)
    # the update is at most ~lr in magnitude; fp32 evaluation of m/(sqrt(v)+eps) is good to ~1e-6 relative
    np.testing.assert_allclose(dp.cpu().numpy(), ep, rtol=0, atol=5e-7)  # half an ulp of |p| < 8, plus the update
    assert np.array_equal(dp.cpu().numpy()[:100], p[:100]) or t > 1  # zero gradient, zero moments: no move


HP_SMALL = {"use_color": 1, "batch_size": 2, "learning_rate": 0.001, "decay_step": 200000,
            "learning_rate_decay_rate": 0.7, "bn_init_decay": 0.5, "bn_decay_decay_rate": 0.5,
            "bn_decay_clip": 0.99, "l1_npoint": 256, "l1_radius": 0.1, "l1_nsample": 32, "l2_npoint": 64,
            "l2_radius": 0.2, "l2_nsample": 32, "l3_npoint": 16, "l3_radius": 0.4, "l3_nsample": 32,
            "l4_npoint": 8, "l4_radius": 0.8, "l4_nsample": 32}


def small_batches(count, b=2, n=1024, seed=100):
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(count):
        pc = np.concatenate([rs.random_sample((b, n, 3)), rs.random_sample((b, n, 3))], -1).astype(np.float32)
        labels = rs.randint(0, 9, (b, n)).astype(np.int32)
        smpw = rs.uniform(0.5, 2.0, (b, n)).astype(np.float32)
        out.append((pc, labels, smpw))
    return out


def load_oracle_params(tr, params):
    sd = {}
    for k, v in params.items():
        if k.endswith("/weights"):
            v = v.reshape((1,) + v.shape) if k.split("/")[0] in ("fc1", "fc2") else v.reshape((1, 1) + v.shape)
        sd[k] = v
    tr.store.load_state_dict(sd)


def test_two_training_steps_match_oracle(cuda):
    """Trainer.step twice, every step verified from the GPU's OWN state before it (so fp32-vs-fp64 drift
    cannot accumulate into the check): loss against the fp64 oracle on the same weights and dropout mask
    (seed host_seed + k); every parameter gradient strictly (the oracle differentiates with the GPU's ReLU
    masks / pooling winners); the Adam update against the fp64 TF-Adam formula applied to the GPU's
    gradient and moments; BatchNorm moving statistics after exactly ONE EMA update per step (the variable-
    creating pass leaves no trace)."""
    import torch
    import pn2_b200  # noqa: F401
    from pn2_b200.train_step import Trainer
    from pn2_b200.util import tf_util
    from oracle import layers_ref as lr
    hp = HP_SMALL
    (pc, labels, smpw), = small_batches(1)
    b, n = pc.shape[:2]
    params = lr.init_model_params(hp, 9, seed=1)
    tr = Trainer(hp, 9, device="cuda", seed=0, world_size=1)
    load_oracle_params(tr, params)
    seed0 = 1234
    tf_util.set_dropout_seed(seed0)
    d_pc, d_lab, d_w = to_cuda(pc), to_cuda(labels), to_cuda(smpw)
    lr_f, b1, b2, eps = (float(np.float32(x)) for x in (1e-3, 0.9, 0.999, 1e-8))
    for step in (1, 2):
        before = {k: v.reshape(params[k].shape) for k, v in tr.store.state_dict().items()}
        m0 = tr.m.cpu().numpy().astype(np.float64) if tr.m is not None else None
        v0 = tr.v.cpu().numpy().astype(np.float64) if tr.v is not None else None
        tf_util.debug_capture = {}
        try:
            loss = float(tr.step(d_pc, d_lab, d_w).item())
            dec = {k: v.cpu().numpy() for k, v in tf_util.debug_capture.items()}
        finally:
            tf_util.debug_capture = None
        mask = tf_util.dropout_mask(b * n * 128, 0.5, seed0 + step).cpu().numpy().reshape(b, n, 128)
        ctx = lr.Ctx(before, is_training=True, bn_decay=0.5, dropout_masks={"dp1": mask.astype(np.float64)},
                     decisions=dec)
        e_loss = lr.get_loss(lr.get_model(ctx, pc, 9, hp), labels, smpw)
        e_loss.backward()
        assert abs(loss - e_loss.item()) < 5e-5, (step, loss, e_loss.item())
        ours = {k: v.grad.detach().cpu().numpy() for k, v in tr.store.vars.items() if v.trainable}
        bad = lr.compare_grads(ctx, ours, rtol_max=5e-5)  # whole network: see tests/test_layers_gpu.py
        assert not bad, "step %d: " % step + "; ".join(bad)
        after = tr.store.state_dict()
        off = 0
        for v in tr.store.trainable():
            cnt = v.data.numel()
            g = ours[v.name].reshape(-1).astype(np.float64)
            mm = m0[off:off + cnt] if m0 is not None else np.zeros(cnt)
            vv = v0[off:off + cnt] if v0 is not None else np.zeros(cnt)
            exp, _, _ = adam_reference(before[v.name].reshape(-1).astype(np.float64), g, mm, vv, lr_f, b1, b2, eps,
                                       step, 1.0)
            np.testing.assert_allclose(after[v.name].reshape(-1), exp, rtol=0, atol=5e-7,
                                       err_msg="%s step %d" % (v.name, step))
            off += cnt
        for k, mv in ctx.new_moving.items():
            np.testing.assert_allclose(after[k].reshape(mv.shape), mv, rtol=1e-5, atol=1e-5,
                                       err_msg="%s step %d" % (k, step))
    torch.cuda.synchronize()


def _run_steps(mode, batches, seed0=77, hp=None, **trainer_kw):
    """len(batches) steps on a fresh Trainer (same initial weights every time): 'eager' | 'graph' | 'staged' |
    'ahead' | 'ahead_staged'."""
    hp = hp or HP_SMALL
    import torch
    from pn2_b200.train_step import Trainer
    from pn2_b200.util import tf_util
    from oracle import layers_ref as lr
    ahead = mode.startswith("ahead")
    tr = Trainer(hp, 9, device="cuda", seed=0, world_size=1, geometry_ahead=ahead, **trainer_kw)
    load_oracle_params(tr, lr.init_model_params(hp, 9, seed=1))
    tf_util.set_dropout_seed(seed0)
    dev = [tuple(to_cuda(x) for x in bt) for bt in batches]
    losses, moving1 = [], None
    if ahead:
        tr.prime(*dev[0])
    if mode != "eager":
        assert tr.capture(*dev[0]), tr._capture_error
        assert tr.launches_per_replay > 100
    if mode in ("staged", "ahead_staged"):
        host = [tuple(torch.as_tensor(x).pin_memory() for x in bt) for bt in batches]
        tr.stage(*host[1 if ahead else 0])
    for i in range(len(batches)):
        nxt = min(i + 1, len(batches) - 1)  # ahead modes: the batch whose geometry step i computes
        if mode == "eager":
            loss = tr.step(*dev[i])
        elif mode == "graph":
            loss = tr.step_graph(*dev[i])
        elif mode == "ahead":
            loss = tr.step_graph(*dev[nxt])
        elif mode == "ahead_staged":
            loss = tr.step_graph()
            tr.stage(*host[min(nxt + 1, len(batches) - 1)])
        else:
            loss = tr.step_graph()
            if i + 1 < len(batches):
                tr.stage(*host[i + 1])
        losses.append(float(loss.item()))
        if i == 0:
            moving1 = {k: v.copy() for k, v in tr.store.state_dict().items() if "moving" in k}
    torch.cuda.synchronize()
    return losses, moving1, tr.store.state_dict(), tr


def test_graph_replay_matches_eager_steps(cuda):
    """Trainer.capture() must succeed, and 3 step_graph() steps (device inputs, and the staged pinned-host
    feed) must train like 3 eager step() steps: same loss sequence, same weights, same moving statistics --
    within the run-to-run noise of the eager path itself (fp32 atomics order), measured by a second eager run.
    After step 1 the moving statistics must be IDENTICAL in all modes: capture's warm-up passes and its
    validation replay leave no EMA update behind."""
    import pn2_b200  # noqa: F401
    batches = small_batches(3)
    l_a, mv_a, w_a, _ = _run_steps("eager", batches)
    l_b, mv_b, w_b, _ = _run_steps("eager", batches)
    l_g, mv_g, w_g, tr = _run_steps("graph", batches)
    l_s, mv_s, w_s, _ = _run_steps("staged", batches)
    assert tr._graph is not None and tr._capture_error is None
    noise_l = max(abs(a - b) for a, b in zip(l_a, l_b))
    noise_w = max(float(np.abs(w_a[k] - w_b[k]).max()) for k in w_a)
    print("eager-vs-eager noise: loss %.3g weights %.3g; losses eager %s graph %s staged %s"
          % (noise_l, noise_w, l_a, l_g, l_s))
    # Step 1 is deterministic up to fp32 atomics order (1e-7 relative): tight.  From step 2 on, Adam turns the
    # sign of every near-zero gradient into a +-lr move, so two runs of the SAME eager code already differ by
    # ~1.5 lr in some weights and ~1e-4 in the loss after three steps (measured on B200: 2.7e-5 .. 2e-4): the
    # later steps are bounded by what a real defect would exceed by an order of magnitude (a stale batch, a
    # repeated dropout mask or a missing update moves the loss by >= 1e-2), not by that noise.
    for name, (l_x, mv_x, w_x) in {"eager2": (l_b, mv_b, w_b), "graph": (l_g, mv_g, w_g),
                                   "staged": (l_s, mv_s, w_s)}.items():
        assert abs(l_x[0] - l_a[0]) < 2e-6, (name, l_x, l_a)
        for k in mv_a:
            np.testing.assert_allclose(mv_x[k], mv_a[k], rtol=1e-6, atol=1e-7, err_msg="%s %s" % (name, k))
        assert max(abs(a - b) for a, b in zip(l_x, l_a)) <= 2e-3, (name, l_x, l_a, noise_l)
        dw = max(float(np.abs(w_x[k] - w_a[k]).max()) for k in w_a)
        # Adam's m/sqrt(v) can exceed 1 after the first step: a sign-flipped near-zero gradient moves a weight by a few
        # lr per step in either run (measured 2.6e-3 .. 7.1e-3 between identical eager runs); real defects are O(0.1)
        assert dw <= 2e-2, (name, dw, noise_w)
    # a defect of the kind this test exists for: the same batch replayed (inputs not refreshed) is far outside
    l_stale = [l_a[0]] * 3
    assert max(abs(a - b) for a, b in zip(l_stale, l_a)) > 1e-2


def test_geometry_ahead_trains_like_the_plain_graph_steps(cuda):
    """Trainer(geometry_ahead=True): every replay runs the dense stage of the batch loaded one call earlier and, on
    a second stream of the same graph, the sampling / neighbour search of the batch handed in.  4 steps on 4
    different batches must train like 4 plain graph steps.  The learning rate sits at the schedule's floor (1e-5),
    so the chaotic part of graph-vs-eager above (Adam turning the sign of near-zero gradients into +-lr moves) is
    100x smaller and the bound can be tight at EVERY step: a dense stage fed with the geometry, the colours, the
    labels or the dropout mask of the wrong batch moves the loss by > 1e-3 (checked at the end).  The tape left behind must be
    bit-identical to the geometry of the last batch handed in, and the SM budget of the persistent kernels must be
    back at the whole device."""
    import torch
    import pn2_b200  # noqa: F401
    from pn2_b200 import _ffi, model
    hp = dict(HP_SMALL, learning_rate=1e-5)
    batches = small_batches(4)
    l_g, mv_g, w_g, _ = _run_steps("graph", batches, hp=hp)
    l_h, _, w_h, _ = _run_steps("graph", batches, hp=hp)
    noise = max(abs(a - b) for a, b in zip(l_g, l_h))
    for mode in ("ahead", "ahead_staged"):
        l_x, mv_x, w_x, tr = _run_steps(mode, batches, hp=hp)
        assert tr._graph is not None and tr._capture_error is None
        print("losses graph %s %s %s (graph-vs-graph noise %.3g)" % (l_g, mode, l_x, noise))
        assert abs(l_x[0] - l_g[0]) < 2e-6, (mode, l_x, l_g)
        for k in mv_g:
            np.testing.assert_allclose(mv_x[k], mv_g[k], rtol=1e-6, atol=1e-7, err_msg="%s %s" % (mode, k))
        assert max(abs(a - b) for a, b in zip(l_x, l_g)) <= 1e-4, (mode, l_x, l_g, noise)
        dw = max(float(np.abs(w_x[k] - w_g[k]).max()) for k in w_g if "moving" not in k)
        assert dw <= 1e-4, (mode, dw)  # 4 steps x (at most ~2 lr per sign flip)
        fresh = model.get_geometry(to_cuda(batches[-1][0]), hp)
        assert len(fresh.tensors()) == len(tr._tape.tensors()) == 16
        for a, b in zip(tr._tape.tensors(), fresh.tensors()):
            assert a.dtype == b.dtype and torch.equal(a, b)
        assert _ffi.lib().pn2_get_sm_budget() == torch.cuda.get_device_properties(0).multi_processor_count
    # the batches differ enough for a mix-up to show: every pair of step losses is >= 10x the bound apart
    assert min(abs(a - b) for i, a in enumerate(l_g) for b in l_g[i + 1:]) > 1e-3, l_g


def test_weight_gradients_on_a_second_stream_train_alike(cuda):
    """Trainer(wgrad_sms=k): every pn2_linear_wgrad of the backward pass runs on a second stream (k SMs for its
    persistent kernel) next to the input-gradient / BatchNorm-backward chain.  Same gradients, so 4 steps at the
    learning-rate floor must match the single-stream trainer at every step -- eagerly, by graph replay, and combined
    with the geometry-ahead mode; a weight gradient read before it is complete (a missing join) or computed from a
    recycled buffer would move the weights and with them the next losses."""
    import pn2_b200  # noqa: F401
    hp = dict(HP_SMALL, learning_rate=1e-5)
    batches = small_batches(4)
    l_g, mv_g, w_g, _ = _run_steps("graph", batches, hp=hp, wgrad_sms=0)
    for mode in ("eager", "graph", "ahead"):
        l_x, mv_x, w_x, tr = _run_steps(mode, batches, hp=hp, wgrad_sms=48)
        assert tr.wgrad_sms == 48 and tr._wstream is not None
        print("losses single-stream %s, wgrad stream (%s) %s" % (l_g, mode, l_x))
        assert max(abs(a - b) for a, b in zip(l_x, l_g)) <= 1e-4, (mode, l_x, l_g)
        assert abs(l_x[0] - l_g[0]) < 2e-6, (mode, l_x, l_g)
        dw = max(float(np.abs(w_x[k] - w_g[k]).max()) for k in w_g if "moving" not in k)
        assert dw <= 1e-4, (mode, dw)


def test_eager_step_after_capture_draws_fresh_dropout_masks(cuda):
    """ADVICE r1: with a captured graph installed, eager step() must still advance the dropout counter
    (and re-capture must not rewind it): four steps -> four different masks -> four different losses on
    the same batch with a zero learning rate."""
    import pn2_b200  # noqa: F401
    from pn2_b200.train_step import Trainer
    hp = dict(HP_SMALL, learning_rate=0.0)
    (pc, labels, smpw), = small_batches(1)
    d = tuple(to_cuda(x) for x in (pc, labels, smpw))
    tr = Trainer(hp, 9, device="cuda", seed=0, world_size=1)
    assert tr.capture(*d), tr._capture_error
    losses = [float(tr.step_graph(*d).item()), float(tr.step(*d).item())]
    assert tr.capture(*d), tr._capture_error
    losses += [float(tr.step_graph(*d).item()), float(tr.step(*d).item())]
    assert int(tr._seed_dev.item()) == 4
    assert len({round(x, 7) for x in losses}) == 4, losses


def test_data_parallel_two_ranks_nccl(cuda):
    """2 ranks x NCCL (needs 2 GPUs): replicas start from rank 0's weights, the reduced gradient equals the
    mean of the shard gradients, and the weights stay identical across ranks after 2 steps."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29561", os.path.join(root, "tests", "dp_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0 and out.stdout.count("DP_OK") == 2, out.stdout[-3000:] + out.stderr[-3000:]


def test_loss_with_out_of_range_label_is_nan_not_garbage(cuda):
    """ADVICE r1: a label outside [0, C) must not index the logits out of bounds; like TF's GPU kernel the
    row's loss (and gradient) is NaN, everything else stays finite."""
    import torch
    import pn2_b200  # noqa: F401
    from pn2_b200 import model
    rs = np.random.RandomState(0)
    pred = to_cuda(rs.normal(size=(2, 64, 9)).astype(np.float32)).requires_grad_(True)
    lab = rs.randint(0, 9, (2, 64)).astype(np.int32)
    good = model.get_loss(pred, to_cuda(lab), to_cuda(np.ones((2, 64), np.float32)))
    assert np.isfinite(good.item())
    lab[1, 5] = 9
    lab[0, 7] = -1
    bad = model.get_loss(pred, to_cuda(lab), to_cuda(np.ones((2, 64), np.float32)))
    assert np.isnan(bad.item())
    bad.backward()
    g = pred.grad.cpu().numpy()
    assert np.isnan(g[1, 5]).all() and np.isnan(g[0, 7]).all()
    g[1, 5] = 0
    g[0, 7] = 0
    assert np.isfinite(g).all()


def test_full_size_step_properties(cuda):
    """BASELINE.json configs[1] at its FULL size (16 clouds x 8192 points, semantic.json): the oracle cannot
    follow here in seconds, so the step is pinned by size-independent properties of what it computes --
    (1) the same pass twice gives the same loss and gradient up to the fp32-atomics noise floor,
    (2) linearity in the sample weights (SUM_BY_NONZERO_WEIGHTS: doubling every weight doubles loss and gradient
        exactly, up to that floor),
    (3) the captured graph reproduces the eager pass on the same weights and the same dropout counter,
    (4) clouds whose weights are all zero contribute nothing: their labels can be anything."""
    import pn2_b200  # noqa: F401
    import bench
    from pn2_b200.train_step import Trainer
    pc, labels, smpw = bench.make_batch(16, 8192, 100)
    rs = np.random.RandomState(5)
    smpw = rs.uniform(0.5, 2.0, smpw.shape).astype(np.float32)
    smpw[3] = 0.0
    tr = Trainer(bench.HP, bench.NUM_CLASS, device="cuda", seed=0, world_size=1)
    d = [to_cuda(x) for x in (pc, labels, smpw)]

    def fb(inputs):
        loss = float(tr.forward_backward(*inputs).item())
        return loss, tr.grads.clone()

    l0, g0 = fb(d)
    gmax = float(g0.abs().max())
    assert np.isfinite(l0) and bool(g0.isfinite().all()) and gmax > 0
    l1, g1 = fb(d)                                            # (1)
    noise = float((g1 - g0).abs().max())
    assert abs(l1 - l0) < 2e-6 * max(1.0, abs(l0)) and noise < 1e-4 * gmax, (l0, l1, noise, gmax)
    l2, g2 = fb([d[0], d[1], d[2] * 2.0])                     # (2)
    assert abs(l2 - 2 * l0) < 1e-5 * max(1.0, abs(l0)), (l2, l0)
    assert float((g2 - 2 * g0).abs().max()) <= 4 * noise + 1e-6 * gmax
    lab2 = labels.copy()                                      # (4)
    lab2[3] = (lab2[3] + 3) % 9
    l3, g3 = fb([d[0], to_cuda(lab2), d[2]])
    assert abs(l3 - l0) < 2e-6 * max(1.0, abs(l0)), (l3, l0)
    assert float((g3 - g0).abs().max()) <= 4 * noise + 1e-6 * gmax
    assert tr.capture(*d), tr._capture_error                  # (3)
    import torch
    with torch.cuda.stream(tr.stream):                        # one replay WITHOUT the optimizer step (the learning
        tr._seed_dev.add_(1)                                  # rate schedule is clipped at 1e-5, never zero)
        tr._graph.replay()
    tr.stream.synchronize()
    l4, g4 = float(tr._static_loss.item()), tr.grads.clone()
    l5, g5 = fb(d)                                            # eager pass at the same dropout counter
    assert abs(l4 - l5) < 2e-6 * max(1.0, abs(l5)), (l4, l5)
    assert float((g4 - g5).abs().max()) <= 4 * noise + 1e-6 * gmax


def test_full_size_geometry_ahead_replay_equals_the_plain_pass(cuda):
    """BASELINE.json configs[1] at its FULL size, in the mode bench.py times: one geometry-ahead replay (dense stage of
    batch A from its tape, sampling / neighbour search of batch B on the side stream, weight gradients on theirs,
    persistent GEMMs on their SM budgets) must give the loss and the gradient of the plain single-stream eager pass on
    batch A with the same weights and dropout counter, and leave behind the tape of batch B bit-identical to the geometry
    computed in place -- i.e. the overlap changes WHEN things run, not WHAT is computed.
    The reference pass runs its forward GEMMs on the same grid as the overlapped one (16 SMs left free): a CTA's fp32
    partial sums of the BatchNorm statistics depend on which tiles it owns, a scale that lands one ulp elsewhere flips a
    handful of the 33 M ReLU / max-pool decisions of this network, and the gradient moves by 1e-3 of its maximum (measured,
    scripts/diag_overlap_grads.py) -- on equal grids the activations are bit-identical and what remains is the summation
    order of the weight gradients (~1e-6)."""
    import torch
    import pn2_b200  # noqa: F401
    import bench
    from pn2_b200 import model
    from pn2_b200.train_step import Trainer
    A = [to_cuda(x) for x in bench.make_batch(16, 8192, 100)]
    B = [to_cuda(x) for x in bench.make_batch(16, 8192, 1100)]
    plain = Trainer(bench.HP, bench.NUM_CLASS, device="cuda", seed=0, world_size=1, wgrad_sms=0)
    plain.forward_reserve = 16
    plain._seed_dev.add_(1)
    l_ref = float(plain.forward_backward(*A).item())
    g_ref = plain.grads.clone()
    l_ref2 = float(plain.forward_backward(*A).item())
    noise = float((plain.grads - g_ref).abs().max())
    gmax = float(g_ref.abs().max())
    tr = Trainer(bench.HP, bench.NUM_CLASS, device="cuda", seed=0, world_size=1, geometry_ahead=True)
    assert tr.wgrad_sms == 64
    tr.prime(*A)
    assert tr.capture(*A), tr._capture_error
    for a, b in zip(tr.store.state_dict().items(), plain.store.state_dict().items()):
        if "moving" not in a[0]:
            np.testing.assert_array_equal(a[1], b[1], err_msg=a[0])   # same seed -> same initial weights
    with torch.cuda.stream(tr.stream):
        for dst, s in zip(tr._next, B):
            dst.copy_(s)
        tr._seed_dev.add_(1)
        tr._graph.replay()                                        # no optimizer step: compare gradients
    tr.stream.synchronize()
    l_x, g_x = float(tr._static_loss.item()), tr.grads.clone()
    assert abs(l_ref2 - l_ref) < 2e-6 * max(1.0, abs(l_ref))
    assert abs(l_x - l_ref) < 2e-6 * max(1.0, abs(l_ref)), (l_x, l_ref)
    assert float((g_x - g_ref).abs().max()) <= 4 * noise + 1e-5 * gmax, (float((g_x - g_ref).abs().max()), noise, gmax)
    fresh = model.get_geometry(B[0], bench.HP)
    for a, b in zip(tr._tape.tensors(), fresh.tensors()):
        assert torch.equal(a, b)
    for a, b in zip(tr._static, B):                               # the inputs moved up as well
        assert torch.equal(a, b)


def test_weight_gradient_stream_gives_the_same_gradient(cuda):
    """The gradient itself (not its effect through Adam, which at the learning-rate floor hides everything but the
    sign): one eager forward_backward with the weight gradients on their own stream (48 SMs; the whole device) against
    the single-stream pass on the same weights, batch and dropout mask.  The forward GEMMs run on the full grid in both,
    so the activations are bit-identical and only the summation order of the weight gradients differs."""
    import pn2_b200  # noqa: F401
    from pn2_b200.train_step import Trainer
    (pc, labels, smpw), = small_batches(1, b=4, n=2048)
    d = tuple(to_cuda(x) for x in (pc, labels, smpw))
    ref = Trainer(HP_SMALL, 9, device="cuda", seed=0, world_size=1, wgrad_sms=0)
    ref._seed_dev.add_(1)
    l0 = float(ref.forward_backward(*d).item())
    g0 = ref.grads.clone()
    ref.forward_backward(*d)
    noise, gmax = float((ref.grads - g0).abs().max()), float(g0.abs().max())
    assert gmax > 0 and noise < 1e-4 * gmax
    for sms in (48, 148):
        tr = Trainer(HP_SMALL, 9, device="cuda", seed=0, world_size=1, wgrad_sms=sms)
        assert tr._wstream is not None
        tr._seed_dev.add_(1)
        l1 = float(tr.forward_backward(*d).item())
        dg = float((tr.grads - g0).abs().max())
        assert abs(l1 - l0) < 2e-6 * max(1.0, abs(l0)), (sms, l1, l0)
        assert dg <= 4 * noise + 1e-5 * gmax, (sms, dg, noise, gmax)
