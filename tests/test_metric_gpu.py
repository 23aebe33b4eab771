"""GPU: pn2_confusion_from_logits / pn2_confusion_from_labels (csrc/pn2_metrics.cu) against np.argmax + a numpy
bincount and against sklearn / the reference's stored results, compared exactly; util.metric.ConfusionMatrix
inside a captured CUDA graph."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host_confusion(logits, labels, C):
    pd = np.argmax(logits, axis=-1).reshape(-1)
    gt = labels.reshape(-1)
    ok = (gt >= 0) & (gt < C)
    cm = np.bincount(gt[ok] * C + pd[ok], minlength=C * C).reshape(C, C)
    return cm, pd, int((~ok).sum())


def make_case(rows, C, seed):
    """Integer-valued logits (dense ties), NaN / +-inf / all -inf rows, labels including -1 and C."""
    rs = np.random.RandomState(seed)
    x = rs.randint(-3, 4, (rows, C), dtype=np.int8).astype(np.float32)
    if rows:
        k = max(1, rows // 50)
        for kind in range(5):
            r = rs.randint(0, rows, k)
            c = rs.randint(0, C, k)
            if kind == 0:
                x[r, c] = np.nan
            elif kind == 1:  # two NaNs in a row: the first one wins
                x[r, c] = np.nan
                x[r, rs.randint(0, C, k)] = np.nan
            elif kind == 2:
                x[r, c] = np.inf
            elif kind == 3:
                x[r, c] = -np.inf
            else:
                x[r, :] = -np.inf
    labels = rs.randint(-1, C + 1, rows).astype(np.int32)
    return x, labels


def test_numpy_argmax_rule():
    assert np.argmax([1, np.nan, 3, np.nan]) == 1
    assert np.argmax([-np.inf, -np.inf]) == 0
    assert np.argmax([2, 5, 5]) == 1


@pytest.mark.parametrize("C", [1, 2, 9, 13, 64, 128])
@pytest.mark.parametrize("rows", [0, 1, 31, 1000, 16 * 8192, 3 * 2 ** 20 + 7])
def test_confusion_from_logits_matches_numpy(cuda, rows, C):
    import torch
    from pn2_b200.util.metric import ConfusionMatrix
    x, labels = make_case(rows, C, seed=rows + C)
    cm = ConfusionMatrix(C)
    d_x = torch.as_tensor(x).cuda()
    d_l = torch.as_tensor(labels).cuda()
    pred = torch.full((rows,), -7, dtype=torch.int32, device="cuda")
    cm.increment_from_logits(d_x, d_l, pred_out=pred)
    exp_cm, exp_pd, exp_skip = host_confusion(x, labels, C)
    np.testing.assert_array_equal(pred.cpu().numpy(), exp_pd)
    np.testing.assert_array_equal(cm.confusion_matrix, exp_cm)
    assert cm.skipped == exp_skip
    # calls accumulate; a 3-D view and no pred_out
    cm.increment_from_logits(d_x.view(1, rows, C), d_l.view(1, rows))
    cm.increment_from_logits(d_x, d_l)
    np.testing.assert_array_equal(cm.confusion_matrix, 3 * exp_cm)
    assert cm.skipped == 3 * exp_skip
    cm.reset()
    assert cm.confusion_matrix.sum() == 0 and cm.skipped == 0


def test_confusion_from_logits_unaligned_rows(cuda):
    """A logits view that starts 4 bytes into the buffer takes the scalar staging path."""
    import torch
    from pn2_b200.util.metric import ConfusionMatrix
    x, labels = make_case(5000, 9, seed=3)
    buf = torch.empty(x.size + 1, dtype=torch.float32, device="cuda")
    buf[1:] = torch.as_tensor(x.reshape(-1)).cuda()
    d_x = buf[1:].view(5000, 9)
    cm = ConfusionMatrix(9)
    cm.increment_from_logits(d_x, torch.as_tensor(labels).cuda())
    np.testing.assert_array_equal(cm.confusion_matrix, host_confusion(x, labels, 9)[0])


@pytest.mark.parametrize("C,n", [(1, 10), (9, 16 * 8192), (13, 999), (128, 200000)])
def test_confusion_from_labels_matches_sklearn(cuda, C, n):
    import torch
    from sklearn.metrics import confusion_matrix
    from pn2_b200.util.metric import ConfusionMatrix
    rs = np.random.RandomState(C + n)
    gt = rs.randint(-1, C + 1, n)
    pd = rs.randint(-1, C + 1, n)
    cm = ConfusionMatrix(C)
    cm.increment_from_list(gt, pd)  # numpy int64
    cm.increment_from_list(torch.as_tensor(gt.astype(np.int32)).cuda(), torch.as_tensor(pd.astype(np.int32)).cuda())
    exp = confusion_matrix(gt, pd, labels=list(range(C)))
    np.testing.assert_array_equal(cm.confusion_matrix, 2 * exp)
    ok = (gt >= 0) & (gt < C) & (pd >= 0) & (pd < C)
    assert cm.skipped == 2 * int((~ok).sum())
    # labels far outside int32 are dropped, not wrapped into range
    cm.reset()
    cm.increment_from_list(np.array([2 ** 32, 0]), np.array([0, 2 ** 32 + C - 1]))
    assert cm.confusion_matrix.sum() == 0 and cm.skipped == 2


def test_confusion_from_labels_matches_the_reference(cuda):
    from pn2_b200.util.metric import ConfusionMatrix
    with open(os.path.join(ROOT, "tests", "golden", "reference_metrics.json")) as f:
        cases = json.load(f)["increment_from_list"]
    for case in cases:
        gt, pd = np.array(case["gt"]), np.array(case["pd"])
        cm = ConfusionMatrix(case["num_classes"])
        cm.increment_from_list(gt, pd)
        cm.increment_from_list(gt[::3], pd[::-3])
        np.testing.assert_array_equal(cm.confusion_matrix, np.array(case["matrix"]))


def test_increment_and_reference_getters(cuda):
    """The reference's self-test (metric.py:135-168) through increment()."""
    from pn2_b200.util.metric import ConfusionMatrix
    ref = np.array([[0, 1, 2, 3], [0, 4, 5, 6], [0, 7, 8, 9], [0, 10, 11, 12]])
    cm = ConfusionMatrix(num_classes=4)
    for gt in range(4):
        for pd in range(4):
            for _ in range(ref[gt, pd]):
                cm.increment(gt, pd)
    np.testing.assert_array_equal(cm.confusion_matrix, ref)
    exp = np.array([4.0 / (4 + 7 + 10 + 5 + 6), 8.0 / (5 + 8 + 11 + 7 + 9), 12.0 / (6 + 9 + 12 + 10 + 11)])
    np.testing.assert_allclose(cm.get_per_class_ious(), exp)
    assert cm.get_mean_iou() == np.mean(exp)
    assert cm.get_accuracy() == float(4 + 8 + 12) / ((4 + 12) * 9 / 2)


def test_increment_from_logits_in_a_cuda_graph(cuda):
    """Captured once and replayed K times == K eager calls; the caller's stream, no synchronisation."""
    import torch
    from pn2_b200.util.metric import ConfusionMatrix
    x, labels = make_case(16 * 8192, 9, seed=5)
    d_x, d_l = torch.as_tensor(x).cuda(), torch.as_tensor(labels).cuda()
    pred = torch.empty(len(labels), dtype=torch.int32, device="cuda")
    eager, graphed = ConfusionMatrix(9), ConfusionMatrix(9)
    K = 5
    for _ in range(K):
        eager.increment_from_logits(d_x, d_l, pred_out=pred)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        graphed.increment_from_logits(d_x, d_l)  # warm-up (kernel attributes), then undone
        graphed.reset()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            graphed.increment_from_logits(d_x, d_l, pred_out=pred)
    torch.cuda.current_stream().wait_stream(s)
    assert graphed.confusion_matrix.sum() == 0  # capture does not execute
    for _ in range(K):
        g.replay()
    np.testing.assert_array_equal(graphed.confusion_matrix, eager.confusion_matrix)
    np.testing.assert_array_equal(eager.confusion_matrix, K * host_confusion(x, labels, 9)[0])
    assert graphed.skipped == eager.skipped
