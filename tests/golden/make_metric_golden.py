"""Generates reference_metrics.json: what the reference's util/metric.py computes, for tests/test_metric_cpu.py
and tests/test_metric_gpu.py (the reference is not part of the repository, so they compare with this file).

For each matrix: get_per_class_ious, get_mean_iou, get_accuracy and the exact stdout of print_metrics() (floats
as repr strings, so that equality is exact and nan survives JSON).  The matrices: the self-test of metric.py, a
random 9 x 9 matrix, one with a class whose union is zero, one with predictions in column 0 (the [Warn] line)
and an all-zero one (accuracy nan).  Also a few increment_from_list results on seeded label arrays that hold
-1 and C, which sklearn's confusion_matrix(labels=range(C)) drops.

Run on a CPU machine with numpy and scikit-learn, from the repo root:
  python tests/golden/make_metric_golden.py REFERENCE_DIR
"""
import contextlib
import importlib.util
import io
import json
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def matrices():
    rs = np.random.RandomState(7)
    union_zero = rs.randint(0, 50, (9, 9)).astype(np.int64)
    union_zero[:, 0] = 0
    union_zero[4, :] = 0
    union_zero[:, 4] = 0
    warn = rs.randint(0, 50, (5, 5)).astype(np.int64)
    warn[2, 0] = 3
    return {
        "self_test": np.array([[0, 1, 2, 3], [0, 4, 5, 6], [0, 7, 8, 9], [0, 10, 11, 12]], np.int64),
        "random_9": np.concatenate([np.zeros((9, 1), np.int64), rs.randint(0, 5000, (9, 8))], axis=1),
        "union_zero": union_zero,
        "column0_warn": warn,
        "all_zero": np.zeros((9, 9), np.int64),
    }


def label_cases():
    rs = np.random.RandomState(11)
    out = []
    for c, n in ((9, 3000), (4, 300), (13, 4000)):
        gt = rs.randint(-1, c + 1, n)
        pd = rs.randint(-1, c + 1, n)
        out.append((c, gt, pd))
    return out


def main(reference_dir):
    spec = importlib.util.spec_from_file_location("ref_metric", os.path.join(reference_dir, "util", "metric.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    result = {"matrices": {}, "increment_from_list": []}
    for name, m in matrices().items():
        cm = ref.ConfusionMatrix(len(m))
        cm.confusion_matrix += m
        rec = {"matrix": m.tolist()}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")  # 0/0 in get_accuracy of the all-zero matrix
            for getter in ("get_per_class_ious", "get_mean_iou", "get_accuracy"):
                buf = io.StringIO()
                with contextlib.redirect_stdout(buf):
                    v = getattr(cm, getter)()
                rec[getter] = [repr(float(x)) for x in v] if isinstance(v, list) else repr(float(v))
                rec[getter + "_stdout"] = buf.getvalue()
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                cm.print_metrics()
            rec["print_metrics"] = buf.getvalue()
        result["matrices"][name] = rec
    for c, gt, pd in label_cases():
        cm = ref.ConfusionMatrix(c)
        cm.increment_from_list(gt, pd)
        cm.increment_from_list(gt[::3], pd[::-3])  # matrices accumulate over calls
        result["increment_from_list"].append({"num_classes": c, "gt": gt.tolist(), "pd": pd.tolist(),
                                              "matrix": cm.confusion_matrix.tolist()})
    with open(os.path.join(HERE, "reference_metrics.json"), "w") as f:
        json.dump(result, f)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
