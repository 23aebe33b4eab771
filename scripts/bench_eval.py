"""Evaluation on the device, measured: prints one JSON line.

  eval          Trainer.evaluate at B = 16 x 8192 with semantic.json (bench.HP), graph replay and eager launches:
                points/s, with a confusion matrix accumulated every call
  confusion     pn2_confusion_from_logits at (16*8192, 9) and (64*8192, 9): CUDA-event time per call, the byte
                model rows*(4C + 4) read + 4*rows pred_out written, and the rate it implies
  host_path     what the kernel replaces (train.py:246-251): logits device -> host, np.argmax,
                sklearn.metrics.confusion_matrix, at (16*8192, 9)
  train_step    step_graph in geometry-ahead mode with Trainer.train_confusion off and on, alternated step by step in
                one run (the difference is one extra launch in the step graph)
  card          name and power limit of the GPU, read in the same run

Every shape is warmed first; a 256 MB write flushes L2 between timed passes, as in bench.py.  Writes nothing.
  python scripts/bench_eval.py [--steps 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import HP, NUM_CLASS, NBATCH, make_batch  # noqa: E402

HBM_DATASHEET_BPS = 7.7e12  # HGX B200 data sheet, one GPU


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0), "power_limit_w": "not measured"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        lim, clk = (x.strip() for x in q.stdout.strip().split(","))
        out["power_limit_w"], out["max_sm_clock_mhz"] = float(lim), float(clk)
    except Exception as e:  # noqa: BLE001 - report, do not guess
        out["power_limit_error"] = repr(e)
    return out


def timed(fn, reps, flush):
    """CUDA-event time of fn() per call (ms), L2 flushed before every call, outside the events."""
    import torch
    ms = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), float(np.min(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    from sklearn.metrics import confusion_matrix
    import pn2_b200  # noqa: F401
    from pn2_b200.train_step import Trainer
    from pn2_b200.util.metric import ConfusionMatrix
    assert torch.cuda.is_available(), "bench_eval.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    b, n = HP["batch_size"], HP["num_point"]
    batches = [tuple(torch.as_tensor(x).to(dev) for x in make_batch(b, n, 100 + 1000 * j)) for j in range(NBATCH)]
    result = {"card": card(), "config": "semantic.json, B=%d x N=%d, %d classes" % (b, n, NUM_CLASS),
              "l2": "256 MB flush write before every timed call"}

    # ---- Trainer.evaluate ------------------------------------------------------------------------------
    tr = Trainer(HP, NUM_CLASS, device=dev, seed=0)
    cm = ConfusionMatrix(NUM_CLASS)
    ev = {}
    for name, graph in (("graph", True), ("eager", False)):
        for i in range(max(args.warmup, 2)):
            tr.evaluate(*batches[i % NBATCH], confusion=cm, graph=graph)
        k = [0]

        def one():
            tr.evaluate(*batches[k[0] % NBATCH], confusion=cm, graph=graph)
            k[0] += 1
        med, best = timed(one, args.steps, flush)
        ev[name] = {"ms_per_call_median": med, "ms_per_call_min": best, "points_per_s": b * n / (med * 1e-3)}
    ev["graph_capture_error"] = tr._eval_capture_error
    result["eval"] = ev

    # ---- the kernel alone -----------------------------------------------------------------------------------
    conf = {}
    for rows in (16 * 8192, 64 * 8192):
        rs = np.random.RandomState(rows)
        logits = torch.as_tensor(rs.standard_normal((rows, NUM_CLASS)).astype(np.float32)).to(dev)
        labels = torch.as_tensor(rs.randint(0, NUM_CLASS, rows).astype(np.int32)).to(dev)
        pred = torch.empty(rows, dtype=torch.int32, device=dev)
        c = ConfusionMatrix(NUM_CLASS)
        for _ in range(3):
            c.increment_from_logits(logits, labels, pred_out=pred)
        reps = max(args.steps, 50)
        med, best = timed(lambda: c.increment_from_logits(logits, labels, pred_out=pred), reps, flush)
        nbytes = rows * (4 * NUM_CLASS + 4) + 4 * rows
        conf["rows_%d" % rows] = {
            "us_per_call_median": med * 1e3, "us_per_call_min": best * 1e3, "bytes": nbytes,
            "achieved_bytes_per_s": nbytes / (med * 1e-3),
            "datasheet_hbm_floor_us": nbytes / HBM_DATASHEET_BPS * 1e6,
            "note": "one launch between two CUDA events: includes launch latency"}
    result["confusion_from_logits"] = conf

    # ---- the host path it replaces ----------------------------------------------------------------------
    rows = b * n
    rs = np.random.RandomState(1)
    logits = torch.as_tensor(rs.standard_normal((b, n, NUM_CLASS)).astype(np.float32)).to(dev)
    gt = rs.randint(0, NUM_CLASS, (b, n))
    host = {}
    for phase in ("warm", "timed"):
        t0 = time.perf_counter()
        h = logits.cpu().numpy()
        t1 = time.perf_counter()
        pd = np.argmax(h, 2)
        t2 = time.perf_counter()
        confusion_matrix(gt.flatten(), pd.flatten(), labels=list(range(NUM_CLASS)))
        t3 = time.perf_counter()
        host = {"d2h_ms": (t1 - t0) * 1e3, "argmax_ms": (t2 - t1) * 1e3, "sklearn_confusion_ms": (t3 - t2) * 1e3,
                "total_ms": (t3 - t0) * 1e3, "rows": rows}
    result["host_path"] = host

    # ---- the training step with train_confusion off / on, alternated --------------------------------------
    del tr
    torch.cuda.synchronize()
    trainers = {}
    for name in ("off", "on"):
        t = Trainer(HP, NUM_CLASS, device=dev, seed=0, geometry_ahead=True)
        if name == "on":
            t.train_confusion = ConfusionMatrix(NUM_CLASS)
        t.prime(*batches[0])
        for i in range(max(args.warmup, 3)):
            t.step_graph(*batches[(i + 1) % NBATCH])
        trainers[name] = t
    times = {"off": [], "on": []}
    for i in range(args.steps):
        for name in (("off", "on") if i % 2 == 0 else ("on", "off")):
            t = trainers[name]
            flush.zero_()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            t.step_graph(*batches[(i + 1) % NBATCH])
            e.record()
            e.synchronize()
            times[name].append(a.elapsed_time(e))
    result["train_step"] = {
        name: {"ms_median": float(np.median(v)), "ms_min": float(np.min(v)),
               "launches_per_replay": trainers[name].launches_per_replay} for name, v in times.items()}
    result["train_step"]["on_minus_off_ms_median"] = (result["train_step"]["on"]["ms_median"]
                                                      - result["train_step"]["off"]["ms_median"])
    print(json.dumps(result))


if __name__ == "__main__":
    main()
