"""CPU: the host side of util/metric.py against what the reference's metric.py computes
(tests/golden/reference_metrics.json, written by tests/golden/make_metric_golden.py), and the argument checks of
the two evaluation entry points, which run before any CUDA call."""
import contextlib
import ctypes
import io
import json
import os
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_metrics.json")
LIB = os.path.join(ROOT, "open3d-pointnet2-semantic3d_b200", "lib", "libpn2_b200.so")


def golden():
    with open(GOLDEN) as f:
        return json.load(f)


def run(fn, *args):
    buf = io.StringIO()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # 0/0 of the all-zero matrix, as in the reference
        with contextlib.redirect_stdout(buf):
            v = fn(*args)
    return v, buf.getvalue()


@pytest.mark.parametrize("name", ["self_test", "random_9", "union_zero", "column0_warn", "all_zero"])
def test_host_metrics_equal_the_reference(name):
    from pn2_b200.util import metric
    rec = golden()["matrices"][name]
    m = np.array(rec["matrix"], np.int64)
    ious, out = run(metric.get_per_class_ious, m)
    assert [repr(float(x)) for x in ious] == rec["get_per_class_ious"]  # exact: same operations, same order
    assert out == rec["get_per_class_ious_stdout"]
    miou, out = run(metric.get_mean_iou, m)
    assert repr(float(miou)) == rec["get_mean_iou"] and out == rec["get_mean_iou_stdout"]
    acc, out = run(metric.get_accuracy, m)
    assert repr(float(acc)) == rec["get_accuracy"] and out == rec["get_accuracy_stdout"]
    _, out = run(metric.print_metrics, m)
    assert out == rec["print_metrics"]


def test_golden_covers_the_special_cases():
    g = golden()["matrices"]
    assert g["all_zero"]["get_accuracy"] == "nan"
    assert g["column0_warn"]["get_per_class_ious_stdout"].startswith("[Warn] Contains prediction of label 0:")
    m = np.array(g["union_zero"]["matrix"])[1:, 1:]
    assert (m[3, :].sum() + m[:, 3].sum()) == 0 and g["union_zero"]["get_per_class_ious"][3] == "0.0"


def test_print_metrics_labels_length():
    from pn2_b200.util import metric
    with pytest.raises(ValueError, match="len\\(labels\\) != self.num_classes"):
        metric.print_metrics(np.zeros((3, 3), np.int64), labels=["a", "b"])


def test_increment_value_errors():
    from pn2_b200.util.metric import ConfusionMatrix
    cm = ConfusionMatrix.__new__(ConfusionMatrix)  # the checks come before any device work
    cm.num_classes, cm.valid_labels = 4, set(range(4))
    with pytest.raises(ValueError, match="^Invalid value for gt_label$"):
        cm.increment(4, 1)
    with pytest.raises(ValueError, match="^Invalid value for gt_label$"):
        cm.increment(-1, 1)
    with pytest.raises(ValueError, match="^Invalid value for pd_label$"):
        cm.increment(1, 4)


def test_cpu_device_is_rejected():
    from pn2_b200.util.metric import ConfusionMatrix
    with pytest.raises(ValueError, match="no CPU fallback"):
        ConfusionMatrix(9, device="cpu")


def test_validation_without_gpu():
    """Argument checks of pn2_confusion_from_logits / _from_labels happen before any CUDA call."""
    import __graft_entry__ as g
    if not os.path.exists(LIB):
        g.build()
    lib = ctypes.CDLL(LIB)
    vp = ctypes.c_void_p
    f = lib.pn2_confusion_from_logits
    f.argtypes = [ctypes.c_long, ctypes.c_int] + [vp] * 6
    dummy = vp(0x1000)  # never dereferenced: every call below is rejected first
    assert f(8, 0, dummy, dummy, dummy, dummy, None, None) == -1
    assert f(-1, 9, dummy, dummy, dummy, dummy, None, None) == -1
    assert f(8, 129, dummy, dummy, dummy, dummy, None, None) == -3
    assert f(8, 9, dummy, dummy, None, dummy, None, None) == -4
    assert f(8, 9, None, dummy, dummy, dummy, None, None) == -4
    assert f(8, 9, dummy, dummy, dummy, None, None, None) == -4
    assert f(0, 9, None, None, None, None, None, None) == 0  # nothing to count
    h = lib.pn2_confusion_from_labels
    h.argtypes = [ctypes.c_long, ctypes.c_int] + [vp] * 5
    assert h(8, 0, dummy, dummy, dummy, dummy, None) == -1
    assert h(-1, 9, dummy, dummy, dummy, dummy, None) == -1
    assert h(8, 129, dummy, dummy, dummy, dummy, None) == -3
    assert h(8, 9, dummy, dummy, None, dummy, None) == -4
    assert h(8, 9, dummy, None, dummy, dummy, None) == -4
    assert h(0, 9, None, None, None, None, None) == 0
