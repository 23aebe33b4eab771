"""CPU: this package's model.py makes exactly the layer calls the reference's OWN model.py makes -- SURVEY.md
section 7 hard part 7.

The reference's model.py, unmodified, was imported through the tensorflow shim (compat/tensorflow.py) and run
on this package's API surface by tests/golden/make_reference_golden.py; the calls it made are stored in
tests/golden/reference_model_calls.json.  The device kernels cannot run here, so the four functions model.py
calls into (pointnet_sa_module, pointnet_fp_module, tf_util.conv1d, tf_util.dropout) and the loss are replaced
by recorders that (1) bind every call against the REAL function's signature (a wrong keyword or a missing
argument fails), (2) log the normalised arguments and tensor shapes, (3) return CPU tensors of the right shapes.
The same recorders run this package's model.py: it must make exactly the stored calls in the same order --
which makes the package's model.py (the one the GPU parity tests cover) call-for-call equivalent to the
reference file."""
import inspect
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_model_calls.json")
HP = {"use_color": 1, "l1_npoint": 32, "l1_radius": 0.5, "l1_nsample": 8, "l2_npoint": 16, "l2_radius": 1.0,
      "l2_nsample": 8, "l3_npoint": 8, "l3_radius": 2.0, "l3_nsample": 4, "l4_npoint": 4, "l4_radius": 4.0,
      "l4_nsample": 4}


def _norm(v):
    """JSON-ready record of an argument: tensors by shape and dtype."""
    import torch
    if isinstance(v, torch.Tensor):
        return ["tensor", list(v.shape), str(v.dtype)]
    if isinstance(v, (list, tuple)):
        return [_norm(x) for x in v]
    return v


def model_calls(model):
    """The calls ``model`` (a module with the reference's model.py interface) makes into the layer API and the
    loss, with the placeholders it declares, as a JSON-ready dict."""
    import torch
    from pn2_b200 import model as ours
    from pn2_b200.util import pointnet_util as pu, tf_util

    log = []

    def recorder(name, real, make_result):
        sig = inspect.signature(real)

        def fn(*a, **kw):
            bound = sig.bind(*a, **kw)          # TypeError on a call the real function would reject
            bound.apply_defaults()
            log.append([name, [[k, _norm(v)] for k, v in bound.arguments.items() if k != "end_points"]])
            return make_result(bound.arguments)
        return fn

    def sa_result(a):
        b = a["xyz"].shape[0]
        return (torch.zeros(b, a["npoint"], 3), torch.zeros(b, a["npoint"], a["mlp"][-1]),
                torch.zeros(b, a["npoint"], a["nsample"], dtype=torch.int32))

    sa = recorder("pointnet_sa_module", pu.pointnet_sa_module, sa_result)
    fp = recorder("pointnet_fp_module", pu.pointnet_fp_module,
                  lambda a: torch.zeros(a["xyz1"].shape[0], a["xyz1"].shape[1], a["mlp"][-1]))
    loss = recorder("get_loss", ours.get_loss, lambda a: torch.zeros(()))
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(pu, "pointnet_sa_module", sa)
        mp.setattr(pu, "pointnet_fp_module", fp)
        mp.setattr(tf_util, "conv1d", recorder("conv1d", tf_util.conv1d,
                                               lambda a: torch.zeros(*a["inputs"].shape[:-1],
                                                                     a["num_output_channels"])))
        mp.setattr(tf_util, "dropout", recorder("dropout", tf_util.dropout, lambda a: a["inputs"]))
        for m in {ours, model}:                     # `from util.pointnet_util import ...`: bound at import time
            mp.setattr(m, "pointnet_sa_module", sa)
            mp.setattr(m, "pointnet_fp_module", fp)
        mp.setattr(ours, "get_loss", loss)          # the shim's tf.losses resolves it at call time
        pc = torch.as_tensor(np.random.RandomState(0).random_sample((2, 64, 6)).astype(np.float32))
        labels = torch.zeros(2, 64, dtype=torch.int32)
        smpw = torch.ones(2, 64)

        # placeholders: dtype/shape records (model.py:12-19)
        pls = model.get_placeholders(64, HP)
        pred, end_points = model.get_model(pc, True, 9, HP, bn_decay=0.5)
        model.get_loss(pred, labels, smpw, end_points)
        out = {"placeholders": [[list(p.shape), str(p.dtype)] for p in pls], "pred": _norm(pred),
               "end_points": {k: _norm(v) for k, v in sorted(end_points.items())}, "calls": list(log)}
        assert torch.equal(end_points["l0_xyz"], pc[:, :, :3])  # tf.slice

        # use_color = 0 (semantic_no_color.json): no slicing, points=None into layer1
        del log[:]
        model.get_model(pc[:, :, :3].contiguous(), False, 9, dict(HP, use_color=0))
        out["no_color_first_call"] = log[0]
    return json.loads(json.dumps(out))


def test_model_py_makes_the_reference_model_py_calls():
    import pn2_b200  # noqa: F401
    from pn2_b200 import model as ours
    with open(GOLDEN) as f:
        ref = json.load(f)
    got = model_calls(ours)
    assert len(ref["calls"]) == 4 + 4 + 2 + 1 + 1                                     # SA, FP, conv1d, dropout, loss
    assert got["placeholders"] == ref["placeholders"] == [[[None, 64, 6], "torch.float32"],
                                                          [[None, 64], "torch.int32"], [[None, 64], "torch.float32"]]
    assert got["pred"] == ref["pred"] == ["tensor", [2, 64, 9], "torch.float32"]
    assert got["end_points"] == ref["end_points"] and set(ref["end_points"]) == {"l0_xyz", "feats"}
    assert [c[0] for c in got["calls"]] == [c[0] for c in ref["calls"]]
    for a, b in zip(got["calls"], ref["calls"]):
        assert a == b, (a, b)
    first = dict(ref["no_color_first_call"][1])
    assert first["points"] is None and first["xyz"] == ["tensor", [2, 64, 3], "torch.float32"]
    assert got["no_color_first_call"] == ref["no_color_first_call"]
