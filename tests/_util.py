"""Shared helpers for the parity tests."""
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rng_cloud(seed, b, n, scale=(1.0, 1.0, 1.0), shift=(0.0, 0.0, 0.0)):
    """np.random.seed(seed) legacy stream, uniform fp32 like the reference tests
    (tf_ops/test_tf_ops.py:12-15)."""
    rs = np.random.RandomState(seed)
    x = rs.random_sample((b, n, 3)).astype(np.float32)
    return (x * np.asarray(scale, np.float32) + np.asarray(shift, np.float32)).astype(np.float32)


def golden(name):
    """Committed fixture tests/golden/<name>.npz (written by tests/golden/make_golden.py)."""
    return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))


def golden_inputs():
    """The seeded inputs make_golden.py froze the oracle outputs on (same draws, same order)."""
    np.random.seed(100)
    target = np.random.random((64, 8192, 3)).astype("float32")
    reference = np.random.random((64, 1024, 3)).astype("float32")
    inp = {"nn_q": np.ascontiguousarray(target[:1, :256]), "nn_known": np.ascontiguousarray(reference[:1])}
    del target, reference
    rs = np.random.RandomState(100)
    inp["xyz"] = rs.random_sample((2, 1024, 3)).astype(np.float32)
    np.random.seed(100)
    tri = np.random.rand(1, 5, 3, 3).astype("float32")
    ta, tb, tc = tri[:, :, 0], tri[:, :, 1], tri[:, :, 2]
    inp["areas"] = np.sqrt((np.cross(tb - ta, tc - ta) ** 2).sum(2) + 1e-9).astype(np.float32)
    inp["r"] = np.random.rand(1, 8192).astype(np.float32)
    rs = np.random.RandomState(100)
    inp["w"] = rs.random_sample((1, 9000)).astype(np.float32)
    inp["sp"] = rs.random_sample((700, 3)).astype(np.float32)
    inp["sl"] = rs.randint(0, 9, 700).astype(np.int32)
    inp["dp"] = rs.random_sample((400, 3)).astype(np.float32)
    return inp


def to_cuda(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


_REFERENCE = {}


def _reference():
    """tests/golden/reference_kernels.{json,npz}: what the reference's own CUDA kernels returned on the inputs of
    tests/test_ops_gpu.py (written by tests/golden/make_reference_golden.py)."""
    if not _REFERENCE:
        base = os.path.join(ROOT, "tests", "golden", "reference_kernels")
        with open(base + ".json") as f:
            _REFERENCE["outputs"] = json.load(f)
        _REFERENCE["samples"] = dict(np.load(base + ".npz"))
    return _REFERENCE


def _host(a):
    return np.ascontiguousarray(a.detach().cpu().numpy() if hasattr(a, "detach") else a)


def digest(a):
    """SHA-256 of an array's bytes (C order)."""
    return hashlib.sha256(_host(a).tobytes()).hexdigest()


def sample_positions(size, count=4096):
    """The fixed flat positions a sampled reference output is stored at."""
    return np.sort(np.random.RandomState(0).choice(size, min(size, count), replace=False))


def assert_reference(key, got):
    """``got`` is bit for bit what the reference's own kernel returned for case ``key`` (stored as shape, dtype
    and SHA-256: the full outputs are too large to commit)."""
    a, exp = _host(got), _reference()["outputs"][key]
    assert [list(a.shape), str(a.dtype)] == [exp["shape"], exp["dtype"]], (key, a.shape, a.dtype, exp)
    assert digest(a) == exp["sha256"], "%s differs from the reference kernel's output" % key


def assert_reference_close(key, got, atol, rtol):
    """``got`` matches the reference kernel's output for case ``key`` within the tolerance, at the stored
    sample of positions (outputs of fp32 atomics: their bits depend on the order of the additions)."""
    a, exp = _host(got), _reference()["outputs"][key]
    assert [list(a.shape), str(a.dtype)] == [exp["shape"], exp["dtype"]], (key, a.shape, a.dtype, exp)
    np.testing.assert_allclose(a.reshape(-1)[sample_positions(a.size)], _reference()["samples"][key],
                               atol=atol, rtol=rtol, err_msg=key)
