"""Generates the fixtures that hold what the reference project itself computes, for the tests that compare
this project with it (the reference is not part of the repository, so they compare with these files):

  reference_kernels.json / .npz  outputs of the reference's own CUDA kernels (oracle/_ref/libref_tfops.so,
                                 built by `make -C oracle REF=<reference checkout>`) on the inputs of
                                 tests/test_ops_gpu.py: shape, dtype and SHA-256 of every output a test
                                 compares bit for bit; a fixed sample (_util.sample_positions) of the
                                 outputs of fp32 atomics, which a test compares within a tolerance
  reference_line_counts.json    lines of every source file of the reference tree (tests/test_citations_cpu.py)
  reference_model_calls.json    the layer calls the reference's model.py makes, imported unmodified through
                                 the tensorflow shim (tests/test_reference_model_dropin_cpu.py)

Run from the repo root:
  python tests/golden/make_reference_golden.py kernels             (on a GPU, after building oracle/_ref)
  python tests/golden/make_reference_golden.py tree REFERENCE_DIR  (no GPU needed)
"""
import ctypes
import glob
import importlib.util
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from _util import digest, rng_cloud, sample_positions, to_cuda  # noqa: E402


class RefKernels:
    """The reference's own CUDA kernels (oracle/_ref/libref_tfops.so, see oracle/ref_shim.cu).  Device
    pointers in, nothing copied."""

    def __init__(self):
        self.lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_tfops.so"))

    @staticmethod
    def _p(t):
        return ctypes.c_void_p(t.data_ptr())

    def _empty(self, shape, dtype, like):
        import torch
        torch.cuda.synchronize()  # the reference launchers run on the legacy default stream
        return torch.empty(shape, dtype=dtype, device=like.device)

    def prob_sample(self, inp, inpr):
        """-> (indices, cdf): tf_sampling.cu:212-216 (cumsumKernel + binarysearchKernel)."""
        import torch
        b, n = inp.shape
        m = inpr.shape[1]
        temp = self._empty((b, n), torch.float32, inp)
        out = self._empty((b, m), torch.int32, inp)
        assert self.lib.ref_prob_sample(b, n, m, self._p(inp), self._p(inpr), self._p(temp), self._p(out), 1) == 0
        return out, temp

    def fps(self, inp, m):
        import torch
        b, n, _ = inp.shape
        temp = self._empty((32, n), torch.float32, inp)
        out = self._empty((b, m), torch.int32, inp)
        assert self.lib.ref_fps(b, n, m, self._p(inp), self._p(temp), self._p(out), 1) == 0
        return out

    def query_ball_point(self, radius, nsample, xyz1, xyz2):
        import torch
        b, n, _ = xyz1.shape
        m = xyz2.shape[1]
        idx = self._empty((b, m, nsample), torch.int32, xyz1)
        cnt = self._empty((b, m), torch.int32, xyz1)
        assert self.lib.ref_query_ball_point(b, n, m, ctypes.c_float(radius), nsample, self._p(xyz1),
                                             self._p(xyz2), self._p(idx), self._p(cnt), 1) == 0
        return idx, cnt

    def group_point(self, points, idx):
        import torch
        b, n, c = points.shape
        _, m, ns = idx.shape
        out = self._empty((b, m, ns, c), torch.float32, points)
        assert self.lib.ref_group_point(b, n, c, m, ns, self._p(points), self._p(idx), self._p(out), 1) == 0
        return out

    def gather_point(self, inp, idx):
        import torch
        b, n, _ = inp.shape
        m = idx.shape[1]
        out = self._empty((b, m, 3), torch.float32, inp)
        assert self.lib.ref_gather_point(b, n, m, self._p(inp), self._p(idx), self._p(out), 1) == 0
        return out

    def selection_sort(self, k, dist):
        """-> (outi, out): the reference's own selection_sort_gpu (tf_grouping.cu:95-136)."""
        import torch
        b, m, n = dist.shape
        outi = self._empty((b, m, n), torch.int32, dist)
        out = self._empty((b, m, n), torch.float32, dist)
        assert self.lib.ref_selection_sort(b, n, m, int(k), self._p(dist), self._p(outi), self._p(out), 1) == 0
        return outi, out

    def gather_point_grad(self, inp, idx, out_g):
        import torch
        b, n, _ = inp.shape
        m = idx.shape[1]
        g = self._empty((b, n, 3), torch.float32, inp)
        assert self.lib.ref_gather_point_grad(b, n, m, self._p(out_g), self._p(idx), self._p(g), 1) == 0
        return g

    def group_point_grad(self, points, idx, grad_out):
        import torch
        b, n, c = points.shape
        _, m, ns = idx.shape
        g = self._empty((b, n, c), torch.float32, points)
        assert self.lib.ref_group_point_grad(b, n, c, m, ns, self._p(grad_out), self._p(idx), self._p(g), 1) == 0
        return g


def kernels():
    import torch
    import test_ops_gpu as t
    ref = RefKernels()
    outputs, samples = {}, {}

    def exact(key, a):
        a = np.ascontiguousarray(a.cpu().numpy())
        outputs[key] = {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": digest(a)}

    def sampled(key, a):
        a = a.cpu().numpy()
        outputs[key] = {"shape": list(a.shape), "dtype": str(a.dtype)}
        samples[key] = a.reshape(-1)[sample_positions(a.size)]

    for key, x, m in t.fps_reference_inputs():
        exact(key, ref.fps(to_cuda(x), m))
    for key, radius, ns, x1, x2 in t.ball_reference_inputs():
        idx, cnt = ref.query_ball_point(radius, ns, to_cuda(x1), to_cuda(x2))
        exact(key + "_cnt", cnt)
        exact(key + "_idx", idx)
    for name, d in sorted(t._selection_cases().items()):
        for k in (1, 16, 128):
            outi, out = ref.selection_sort(k, to_cuda(np.ascontiguousarray(d, np.float32)))
            exact("select_%s_k%d_idx" % (name, k), outi)
            exact("select_%s_k%d_val" % (name, k), out)
    for case in t.KNN_REFERENCE_CASES:
        key, x1, x2 = t.knn_reference_inputs(*case)
        k = case[3]
        outi, out = ref.selection_sort(k, to_cuda(t._sqdist_matrix(x1, x2)))
        exact(key + "_idx", outi[:, :, :k])
        exact(key + "_val", out[:, :, :k])
    x, g, groups = t.gather_group_reference_inputs()
    x = to_cuda(x)
    fps = ref.fps(x, 256)
    exact("gather_point", ref.gather_point(x, fps))
    exact("gather_point_grad", ref.gather_point_grad(x, fps, to_cuda(g)))
    idx, _ = ref.query_ball_point(0.2, 32, x, ref.gather_point(x, fps))
    for c, pts, go in groups:
        pts = to_cuda(pts)
        exact("group_point_c%d" % c, ref.group_point(pts, idx))
        sampled("group_point_grad_c%d" % c, ref.group_point_grad(pts, idx, to_cuda(go)))
    for b, n, m in t.PROB_REFERENCE_CASES:
        ids, cdf = ref.prob_sample(*(to_cuda(a) for a in t._prob_inputs(b, n, m)))
        exact("prob_%d_%d_%d_idx" % (b, n, m), ids)
        exact("prob_%d_%d_%d_cdf" % (b, n, m), cdf)
    exact("fps_cluster_2_30000_256", ref.fps(to_cuda(rng_cloud(77, 2, 30000)), 256))
    torch.cuda.synchronize()
    with open(os.path.join(HERE, "reference_kernels.json"), "w") as f:
        json.dump(outputs, f, indent=1, sort_keys=True)
    np.savez_compressed(os.path.join(HERE, "reference_kernels.npz"), **samples)


def tree(ref_dir):
    lengths = {}
    for p in glob.glob(os.path.join(ref_dir, "**", "*"), recursive=True):
        if os.path.isfile(p) and p.endswith((".cu", ".cpp", ".py", ".json", ".cmake")):
            with open(p, errors="replace") as f:
                n = sum(1 for _ in f)
            name = os.path.basename(p)
            lengths[name] = max(lengths.get(name, 0), n)
    with open(os.path.join(HERE, "reference_line_counts.json"), "w") as f:
        json.dump(lengths, f, indent=1, sort_keys=True)

    import pn2_b200  # noqa: F401
    from pn2_b200.compat import tensorflow as tfs
    from test_reference_model_dropin_cpu import model_calls
    assert tfs.install(), "a real tensorflow is importable here"
    spec = importlib.util.spec_from_file_location("reference_model_py", os.path.join(ref_dir, "model.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)  # `import tensorflow`, `import util.tf_util`, ... resolve to this package
    calls = model_calls(ref)
    assert "classify loss" in tfs.summary.values and len(tfs.get_collection("losses")) >= 1
    with open(os.path.join(HERE, "reference_model_calls.json"), "w") as f:
        json.dump(calls, f, indent=1)


if __name__ == "__main__":
    if sys.argv[1:2] == ["kernels"]:
        kernels()
    elif sys.argv[1:2] == ["tree"] and len(sys.argv) == 3:
        tree(sys.argv[2])
    else:
        sys.exit(__doc__)
    print("wrote fixtures")
