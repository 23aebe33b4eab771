"""GPU: evaluation on the device -- Trainer.evaluate (eval_one_epoch, train.py:263-330), Trainer.train_confusion
(the metrics of train_one_epoch, train.py:234-251) and Predictor.predict_scene (predict.py:146-205), at the
small configuration of tests/test_train_step_gpu.py."""
import contextlib

import numpy as np
import pytest

from _util import to_cuda
from test_train_step_gpu import HP_SMALL, load_oracle_params, small_batches

pytestmark = pytest.mark.gpu


def host_confusion(gt, pd, C=9):
    gt, pd = np.asarray(gt).reshape(-1), np.asarray(pd).reshape(-1)
    return np.bincount(gt * C + pd, minlength=C * C).reshape(C, C)


def eval_params(seed=1):
    """Oracle weights with non-trivial BatchNorm affine parameters and moving statistics."""
    from oracle import layers_ref as lr
    rs = np.random.RandomState(seed + 100)
    params = lr.init_model_params(HP_SMALL, 9, seed=seed)
    for k in list(params):
        if k.endswith("moving_mean"):
            params[k] = rs.normal(0, 0.2, params[k].shape).astype(np.float32)
        elif k.endswith("moving_variance"):
            params[k] = rs.uniform(0.5, 2.0, params[k].shape).astype(np.float32)
        elif k.endswith("/bn/gamma"):
            params[k] = rs.uniform(0.5, 1.5, params[k].shape).astype(np.float32)
        elif k.endswith("/bn/beta") or k.endswith("/biases"):
            params[k] = rs.uniform(-0.3, 0.3, params[k].shape).astype(np.float32)
    return params


@contextlib.contextmanager
def recorded_logits(monkeypatch):
    """Wrap model.get_model: the list receives (is_training, logits) of every forward pass.  In graph mode the
    tensor of the captured pass holds the values of the last replay."""
    import pn2_b200.model as model
    seen, inner = [], model.get_model

    def wrapped(point_cloud, is_training, *a, **kw):
        pred, ep = inner(point_cloud, is_training, *a, **kw)
        seen.append((bool(is_training), pred))
        return pred, ep

    monkeypatch.setattr(model, "get_model", wrapped)
    yield seen


def test_evaluate_matches_the_oracle_and_both_modes_agree(cuda, monkeypatch):
    import torch
    from pn2_b200.train_step import Trainer
    from pn2_b200.util.metric import ConfusionMatrix
    from oracle import layers_ref as lr
    params = eval_params()
    (pc, labels, smpw), = small_batches(1, seed=300)
    tr = Trainer(HP_SMALL, 9, device="cuda", seed=0)
    load_oracle_params(tr, params)
    d = tuple(to_cuda(x) for x in (pc, labels, smpw))
    cm_eager, cm_graph = ConfusionMatrix(9), ConfusionMatrix(9)
    with recorded_logits(monkeypatch) as seen:
        loss_eager = tr.evaluate(*d, confusion=cm_eager, graph=False)
        training, logits = seen[-1]
        assert not training
        logits = logits.cpu().numpy()
    e_loss = lr.get_loss(lr.get_model(lr.Ctx(params, is_training=False), pc, 9, HP_SMALL), labels, smpw)
    assert abs(float(loss_eager) - e_loss.item()) < 5e-5, (float(loss_eager), e_loss.item())
    np.testing.assert_array_equal(cm_eager.confusion_matrix, host_confusion(labels, np.argmax(logits, -1)))
    for _ in range(2):  # the first call captures, the second replays
        loss_graph = tr.evaluate(*d, confusion=cm_graph)
    assert tr._eval_capture_error is None, tr._eval_capture_error
    assert len(tr._eval_graphs) == 1 and next(iter(tr._eval_graphs.values())) is not None
    np.testing.assert_array_equal(cm_graph.confusion_matrix, 2 * cm_eager.confusion_matrix)
    assert abs(float(loss_graph) - float(loss_eager)) <= 1e-6 * max(1.0, abs(float(loss_eager)))
    # the returned loss is the call's own: a later evaluation of another batch does not overwrite it
    (pc2, lab2, w2), = small_batches(1, seed=301)
    before = float(loss_graph)
    tr.evaluate(to_cuda(pc2), to_cuda(lab2), to_cuda(w2))
    torch.cuda.synchronize()
    assert float(loss_graph) == before


def state_snapshot(tr):
    import torch
    torch.cuda.synchronize()
    snap = {"flat": tr.flat.clone(), "m": tr.m.clone(), "v": tr.v.clone(), "seed_dev": tr._seed_dev.clone(),
            "step_count": tr.step_count, "graph": tr._graph, "launches": tr.launches_per_replay}
    for k, v in tr.store.vars.items():
        if not v.trainable:
            snap["moving/" + k] = v.data.clone()
    for i, t in enumerate(list(tr._static) + list(tr._next) + tr._tape.tensors()):
        snap["pipeline/%d" % i] = t.clone()
    return snap


def assert_same_state(a, b):
    import torch
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert torch.equal(a[k], b[k]), k
        else:
            assert a[k] is b[k] or a[k] == b[k], k


def test_evaluate_leaves_training_state_untouched(cuda):
    """evaluate() between geometry-ahead step_graph calls: weights, Adam moments, moving statistics, counters,
    the training graph and the _static/_next/_tape pipeline stay bit-identical, and the training graph is not
    re-captured."""
    from pn2_b200.train_step import Trainer
    from pn2_b200.util.metric import ConfusionMatrix
    from oracle import layers_ref as lr
    batches = [tuple(to_cuda(x) for x in bt) for bt in small_batches(4, seed=310)]
    tr = Trainer(dict(HP_SMALL, learning_rate=1e-4), 9, device="cuda", seed=0, geometry_ahead=True)
    load_oracle_params(tr, lr.init_model_params(HP_SMALL, 9, seed=1))
    tr.prime(*batches[0])
    tr.step_graph(*batches[1])
    g0 = tr._graph
    cm = ConfusionMatrix(9)
    (pc, lab, w), = small_batches(1, seed=311)
    for mode in (True, False, True):
        before = state_snapshot(tr)
        tr.evaluate(to_cuda(pc), to_cuda(lab), to_cuda(w), confusion=cm, graph=mode)
        assert_same_state(before, state_snapshot(tr))
    assert tr._eval_capture_error is None, tr._eval_capture_error
    assert cm.confusion_matrix.sum() == 3 * lab.size
    tr.step_graph(*batches[2])
    tr.step_graph(*batches[3])
    assert tr._graph is g0 and tr.step_count == 3


def test_evaluate_before_training_creates_the_variables(cuda):
    from pn2_b200.train_step import Trainer
    (pc, lab, w), = small_batches(1, seed=320)
    tr = Trainer(HP_SMALL, 9, device="cuda", seed=0)
    loss = tr.evaluate(to_cuda(pc), to_cuda(lab), to_cuda(w))
    assert tr.flat is not None and tr.step_count == 0 and np.isfinite(float(loss))
    assert int(tr._seed_dev.item()) == 0
    tr.step(to_cuda(pc), to_cuda(lab), to_cuda(w))
    assert tr.step_count == 1


@pytest.mark.parametrize("mode", ["eager", "graph", "ahead"])
def test_train_confusion_counts_every_training_pass(cuda, monkeypatch, mode):
    """Each pass adds the confusion of its own training-mode logits (dropout applied): B*N counts per step."""
    from pn2_b200.train_step import Trainer
    from pn2_b200.util.metric import ConfusionMatrix
    from oracle import layers_ref as lr
    host = small_batches(4, seed=330)
    batches = [tuple(to_cuda(x) for x in bt) for bt in host]
    tr = Trainer(dict(HP_SMALL, learning_rate=1e-4), 9, device="cuda", seed=0, geometry_ahead=mode == "ahead")
    load_oracle_params(tr, lr.init_model_params(HP_SMALL, 9, seed=1))
    cm = ConfusionMatrix(9)
    tr.train_confusion = cm
    total = np.zeros((9, 9), np.int64)
    with recorded_logits(monkeypatch) as seen:
        if mode == "ahead":
            tr.prime(*batches[0])
        elif mode == "graph":
            assert tr.capture(*batches[0]), tr._capture_error
            assert cm.confusion_matrix.sum() == 0  # warm-up passes and validation replay leave no counts
        for i in range(2):
            if mode == "eager":
                tr.step(*batches[i])
                trained = host[i]
            elif mode == "graph":
                tr.step_graph(*batches[i])
                trained = host[i]
            else:
                tr.step_graph(*batches[i + 1])
                trained = host[i]  # the batch loaded before this call
            training, logits = seen[-1]
            assert training
            step_cm = host_confusion(trained[1], np.argmax(logits.detach().cpu().numpy(), -1))
            total += step_cm
            np.testing.assert_array_equal(cm.confusion_matrix, total)
            assert cm.confusion_matrix.sum() == (i + 1) * trained[1].size
    if mode != "eager":
        assert tr._graph is not None
        counted = tr.launches_per_replay
        tr.train_confusion = None  # clearing re-captures: the graph is today's step again
        tr.step_graph(*batches[3 if mode == "ahead" else 2])
        np.testing.assert_array_equal(cm.confusion_matrix, total)
        assert tr.launches_per_replay == counted - 1
    # eager forward_backward counts too
    tr.train_confusion = cm
    tr.forward_backward(*batches[0])
    assert cm.confusion_matrix.sum() == total.sum() + host[0][1].size


def test_launches_per_replay_unchanged_without_train_confusion(cuda):
    from pn2_b200.train_step import Trainer
    from pn2_b200.util.metric import ConfusionMatrix
    batch = tuple(to_cuda(x) for x in small_batches(1, seed=340)[0])
    fresh = Trainer(HP_SMALL, 9, device="cuda", seed=0)
    assert fresh.capture(*batch), fresh._capture_error
    tr = Trainer(HP_SMALL, 9, device="cuda", seed=0)
    tr.train_confusion = ConfusionMatrix(9)
    assert tr.capture(*batch), tr._capture_error
    assert tr.launches_per_replay == fresh.launches_per_replay + 1
    assert tr.train_confusion.confusion_matrix.sum() == 0  # warm-up and validation replay leave no counts
    tr.train_confusion = None
    assert tr.capture(*batch), tr._capture_error
    assert tr.launches_per_replay == fresh.launches_per_replay


def test_predict_scene(cuda):
    """Predictor.predict_scene on a synthetic ~200 k point scene: sparse points = scene.points[index] exactly,
    labels = arg-max of the eval logits (where the top-2 margin exceeds 1e-3), the matrix = sklearn on (gt,
    labels); then the dense step interpolate_label_with_color -> increment_from_list."""
    import torch
    from sklearn.metrics import confusion_matrix
    from pn2_b200 import model, predict
    from pn2_b200.dataset.semantic_dataset import SemanticFileData
    from pn2_b200.tf_ops.tf_interpolate import interpolate_label_with_color
    from pn2_b200.util import tf_util
    from pn2_b200.util.metric import ConfusionMatrix
    hp = dict(HP_SMALL, num_point=1024)
    rs = np.random.RandomState(350)
    n = 200000
    pts = rs.random_sample((n, 3)) * np.array([4.0, 4.0, 1.0])
    cols = rs.random_sample((n, 3))
    gt_scene = rs.randint(0, 9, n)
    scene = SemanticFileData(pts, gt_scene, cols, 1.0, 1.0)
    p = predict.Predictor(eval_params(), 9, hp)
    cm = ConfusionMatrix(9)
    num_samples, bs, seed = 5, 2, 40
    sp, sl = p.predict_scene(scene, num_samples, batch_size=bs, rng=np.random.RandomState(9), seed=seed,
                             confusion=cm)
    assert sp.shape == (num_samples * 1024, 3) and sp.dtype == np.float64
    assert sl.shape == (num_samples * 1024,) and sl.dtype == np.int64
    # the same batches again
    again = np.random.RandomState(9)
    exp_pts, gts, logits = [], [], []
    tf_util.set_default_store(p.store)
    for i in range(3):
        data, gt, _, index, _ = scene.sample_batch(min(bs, num_samples - i * bs), 1024, rng=again, seed=seed + i)
        exp_pts.append(scene.points[index.reshape(-1).long()].cpu().numpy())
        gts.append(gt.cpu().numpy().reshape(-1))
        with torch.no_grad():
            logits.append(model.get_model(data, False, 9, hp)[0].cpu().numpy().reshape(-1, 9))
    np.testing.assert_array_equal(sp, np.concatenate(exp_pts))
    logits, gt = np.concatenate(logits), np.concatenate(gts)
    top2 = np.sort(logits, -1)[:, -2:]
    sure = (top2[:, 1] - top2[:, 0]) > 1e-3
    assert sure.mean() > 0.9
    np.testing.assert_array_equal(sl[sure], np.argmax(logits, -1)[sure])
    np.testing.assert_array_equal(cm.confusion_matrix, confusion_matrix(gt, sl, labels=list(range(9))))
    # dense evaluation (interpolate.py:119-124): device labels straight into the matrix
    dense = torch.as_tensor(pts[::7].astype(np.float32)).cuda()
    dense_gt = torch.as_tensor(gt_scene[::7].astype(np.int32)).cuda()
    dl, _ = interpolate_label_with_color(torch.as_tensor(sp.astype(np.float32)).cuda(),
                                         torch.as_tensor(sl.astype(np.int32)).cuda(), dense, 3)
    dcm = ConfusionMatrix(9)
    dcm.increment_from_list(dense_gt, dl)
    np.testing.assert_array_equal(dcm.confusion_matrix, confusion_matrix(gt_scene[::7], dl.cpu().numpy(),
                                                                         labels=list(range(9))))
