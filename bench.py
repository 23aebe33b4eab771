#!/usr/bin/env python
"""bench.py -- SA+FP forward+backward throughput (points/s) on B200, next to the reference path
on the host CPU.

  python bench.py --gpus N --steps K --warmup W            our engine (libpn2_b200.so)
  python bench.py --impl reference --steps K --warmup W    reference path on the host cores
  python bench.py ... --dump-outputs DIR                   also write what the last timed step computed
                                                           to DIR/<name>.npy

A "step" is one full training step of the reference's SSG network (model.py:22-161 +
train.py:387-388): 4 SA + 4 FP layers + head, weighted CE loss, backward, Adam -- on a batch of
synthetic clouds with semantic.json's hyper-parameters (BASELINE.json configs[1], SURVEY.md 8d).
At N>1 every rank owns --batch clouds (weak scaling) and the step ends with ONE NCCL all-reduce
over the flat gradient buffer.

Timing: W warm-up steps, then K steps timed with CUDA events on the launching stream, each from
the freshly initialised model (restored, like the L2 flush (256 MB write) between timed steps,
outside the events), barrier + synchronize on both sides, MAX over ranks.  `value` has the
inputs resident in HBM; `e2e` repeats the K steps through the same public API with pinned-host
inputs copied in and the loss read back each step.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sa_fp_fwd_bwd_points_per_sec"
UNIT = "points/s"
NUM_CLASS = 9
HP = {  # semantic.json (reference), verbatim values
    "batch_size": 16, "num_point": 8192, "use_color": 1, "learning_rate": 0.001,
    "decay_step": 200000, "learning_rate_decay_rate": 0.7, "bn_init_decay": 0.5,
    "bn_decay_decay_rate": 0.5, "bn_decay_clip": 0.99,
    "l1_radius": 0.5, "l1_nsample": 32, "l1_npoint": 1024,
    "l2_radius": 1.0, "l2_nsample": 32, "l2_npoint": 256,
    "l3_radius": 2.0, "l3_nsample": 32, "l3_npoint": 64,
    "l4_radius": 4.0, "l4_nsample": 32, "l4_npoint": 16,
}


NBATCH = 4  # distinct batches the timed loops rotate through


def make_batch(b, n, seed):
    """SURVEY.md 8d config 2: xyz uniform in a 10 x 10 x 5 box centred like _center_box
    (semantic_dataset.py:109-121), colours U[0,1), labels 1..8, weights 1."""
    rs = np.random.RandomState(seed)
    xyz = rs.random_sample((b, n, 3)) * np.array([10.0, 10.0, 5.0]) - np.array([5.0, 5.0, 0.0])
    col = rs.random_sample((b, n, 3))
    pc = np.concatenate([xyz, col], -1).astype(np.float32)
    labels = rs.randint(1, 9, (b, n)).astype(np.int32)
    smpw = np.ones((b, n), np.float32)
    return pc, labels, smpw


def workload_name(b, n):
    return ("ssg_semantic_json_train_step_B%d_N%d_xyz3+rgb3 (BASELINE.json configs[1]; the "
            "reference's semantic.json has 3 colour channels, not the 6 BASELINE.json words)" % (b, n))


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_step_factory(sample_b, n):
    import torch
    from oracle import layers_ref as lr
    from oracle import oracle as orc
    # PyTorch-CPU ops on (65k..500k) x (6..512) matrices stop scaling (and then regress) beyond a
    # few tens of threads; 16 was the fastest setting measured on the 128-core GPU host.
    cores = min(os.cpu_count() or 1, int(os.environ.get("PN2_CPU_THREADS", "16")))
    torch.set_num_threads(cores)
    lr.set_dtype(torch.float32)
    threads = min(cores, orc.max_threads())
    # index ops: OpenMP over the batch ("all host cores" variant of BASELINE.md section 3)
    for name in ("farthest_point_sample", "query_ball_point", "three_nn"):
        fn = getattr(orc, name)
        setattr(orc, name, (lambda f: (lambda *a, **k: f(*a, **dict(k, threads=threads))))(fn))
    params = lr.init_model_params(HP, NUM_CLASS, seed=0)
    pc, labels, smpw = make_batch(sample_b, n, 100)

    def step():
        ctx = lr.Ctx(params, is_training=True, bn_decay=0.5)
        pred = lr.get_model(ctx, pc, NUM_CLASS, HP)
        loss = lr.get_loss(pred, labels, smpw)
        loss.backward()
        return float(loss.detach())

    return step, cores


def time_cpu(sample_b, n, steps, warmup):
    step, cores = cpu_step_factory(sample_b, n)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return sample_b * n * steps / dt, dt / steps, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_b = args.batch  # the SAME config as our arm: every cloud of the step, all host threads
    val, sec, cores = time_cpu(sample_b, args.npoint, args.steps, args.warmup)
    sample = ("%d clouds x %d points per step (fwd+bwd of the same SSG network): C oracle "
              "(FPS/ball/3-NN, OpenMP over clouds) + PyTorch-CPU fp32 layers" % (sample_b, args.npoint))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": workload_name(args.batch, args.npoint),
                                        "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region: an in-process NVML polling thread (a step
    takes ~5 ms, so the whole timed region is shorter than one `nvidia-smi -lms` period)."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
               (0x4, "sw_power_cap"))

    def __init__(self, gpu_index):
        import threading
        self.sm, self.mx, self.reasons, self.h = [], None, set(), None
        self._stop = threading.Event()
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes the visible devices; map through CUDA_VISIBLE_DEVICES if it is set
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if gpu_index < len(ids) and ids[gpu_index].isdigit():
                    phys = int(ids[gpu_index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _sample(self):
        try:
            self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            try:
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in self.REASONS:
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _run(self):
        if self.h is None:
            return
        while not self._stop.is_set():
            self._sample()
            time.sleep(0.002)

    def stop(self):
        self._stop.set()
        self.t.join(timeout=2)
        if self.h is not None:
            self._sample()
        out = {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons)}
        if self.sm:
            out["sm_mhz"] = float(np.median(self.sm))
            out["samples"] = len(self.sm)
            out["source"] = "nvml, polled every 2 ms inside the timed region"
        else:  # NVML unavailable: one nvidia-smi query right after the timed region
            try:
                q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm,"
                                    "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                                    "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                   timeout=10).stdout.splitlines()[0].split(",")
                out["sm_mhz"], out["sm_max_mhz"] = float(q[0]), float(q[1])
                out["reasons"] = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown",
                                                     "sw_thermal_slowdown", "sw_power_cap"), q[2:6])
                                  if v.strip().lower().startswith("active")]
                out["source"] = "nvidia-smi, one query right after the timed region"
            except Exception:
                pass
        return out


def fps_stream_bytes(b):
    """SURVEY.md 8d: streaming-model bytes of FPS, B*(npoint-1)*N*20 per SA layer."""
    ns = [HP["num_point"], HP["l1_npoint"], HP["l2_npoint"], HP["l3_npoint"]]
    ms = [HP["l1_npoint"], HP["l2_npoint"], HP["l3_npoint"], HP["l4_npoint"]]
    return [b * (m - 1) * n * 20 for n, m in zip(ns, ms)]


def linear_calls(b):
    """(M, K, N) of every shared-MLP layer of one step (SURVEY.md 3.1 shapes; widths from the product's
    own model.py, 3 colour channels)."""
    from pn2_b200.model import FP_MLPS, SA_MLPS
    n0 = HP["num_point"]
    npts = [n0, HP["l1_npoint"], HP["l2_npoint"], HP["l3_npoint"], HP["l4_npoint"]]
    feat = [3, 64, 128, 256, 512]
    calls = []
    for l in (1, 2, 3, 4):
        m = b * npts[l] * HP["l%d_nsample" % l]
        k = feat[l - 1] + 3
        for n in SA_MLPS[l - 1]:
            calls.append((m, k, n))
            k = n
    up = 512
    for l, lo in zip((1, 2, 3, 4), (3, 2, 1, 0)):
        m = b * npts[lo]
        k = up + feat[lo]
        for n in FP_MLPS[l - 1]:
            calls.append((m, k, n))
            k = n
        up = k
    calls += [(b * n0, 128, 128), (b * n0, 128, NUM_CLASS)]
    return calls


def gemm_flops(b):
    """2*M*K*N of every linear forward call of one step (dgrad and wgrad cost the same each)."""
    return sum(2 * m * k * n for m, k, n in linear_calls(b))


def gemm_bytes(b):
    """ALGORITHMIC HBM bytes of the linear calls of one step: forward reads X[M,K] and writes Y[M,N],
    dgrad reads dY[M,N] and writes dX[M,K] (not needed for the first layer of the network), wgrad reads
    X and dY; weights are negligible and L2 resident."""
    calls = linear_calls(b)
    fwd = sum(4 * m * (k + n) for m, k, n in calls)
    dgr = sum(4 * m * (k + n) for m, k, n in calls[1:])
    wgr = sum(4 * m * (k + n) for m, k, n in calls)
    return fwd, dgr, wgr


def config1_row(dev, reps=30):
    """BASELINE.json configs[0] / BASELINE.md section 3: ONE set-abstraction layer, B=2, N=1024, npoint=256,
    nsample=32, C=3, mlp [32,32,64], train-mode BN, forward + backward -- our engine on the GPU (eager
    launches and CUDA-graph replay) next to the oracle port on the host cores, in the same run."""
    import torch
    from pn2_b200.util import pointnet_util, tf_util
    from oracle import layers_ref as lr
    rs = np.random.RandomState(100)
    xyz = rs.random_sample((2, 1024, 3)).astype(np.float32)
    pts = rs.random_sample((2, 1024, 3)).astype(np.float32)
    old_store = tf_util.default_store()
    store = tf_util.set_default_store(tf_util.VariableStore(device=dev, seed=0))
    stream = torch.cuda.Stream(device=dev)
    row = {"workload": "single SA layer B=2 N=1024 npoint=256 nsample=32 C=3 radius 0.2 mlp [32,32,64], fwd+bwd"}
    try:
        with torch.cuda.stream(stream):
            x = torch.as_tensor(xyz).to(dev)
            p = torch.as_tensor(pts).to(dev).requires_grad_(True)

            def fb():
                store.anchor = torch.zeros(1, device=dev, requires_grad=True)
                p.grad = None
                _, out, _ = pointnet_util.pointnet_sa_module(x, p, 256, 0.2, 32, [32, 32, 64], None, False,
                                                            True, 0.5, "layer1")
                out.sum().backward()
            for _ in range(3):
                fb()
            stream.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fb()
            e1.record()
            e1.synchronize()
            row["gpu_eager_ms"] = e0.elapsed_time(e1) / reps
            try:
                import gc
                gc.collect()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream, capture_error_mode="thread_local"):
                    fb()
                g.replay()
                stream.synchronize()
                e0.record()
                for _ in range(reps):
                    g.replay()
                e1.record()
                e1.synchronize()
                row["gpu_graph_ms"] = e0.elapsed_time(e1) / reps
            except Exception as e:  # noqa: BLE001
                row["gpu_graph_error"] = repr(e)[:300]
                torch.cuda.synchronize()
    finally:
        tf_util.set_default_store(old_store)
    best = min(v for k, v in row.items() if k in ("gpu_eager_ms", "gpu_graph_ms"))
    row["gpu_points_per_sec"] = 2 * 1024 / (best * 1e-3)
    # CPU: the oracle port of the same layer (C oracle index ops + PyTorch-CPU fp32), host cores
    lr.set_dtype(torch.float32)
    params = {}
    k = 6
    for i, n in enumerate([32, 32, 64]):
        lr.init_conv(params, rs, "layer1/conv%d" % i, k, n)
        k = n

    def cpu_fb():
        ctx = lr.Ctx(params, is_training=True, bn_decay=0.5)
        pr = torch.tensor(pts, dtype=torch.float32, requires_grad=True)
        _, feat, _ = lr.sa_module(ctx, xyz, pr, 256, 0.2, 32, [32, 32, 64], "layer1")
        feat.sum().backward()
    cpu_fb()
    t0 = time.perf_counter()
    for _ in range(5):
        cpu_fb()
    cpu_ms = (time.perf_counter() - t0) / 5 * 1e3
    row["cpu_ms"] = cpu_ms
    row["cpu_points_per_sec"] = 2 * 1024 / (cpu_ms * 1e-3)
    row["cpu_threads"] = torch.get_num_threads()
    return row


def cfeat6_line(dev, b, n, steps, warmup, flush, ahead=True):
    """SURVEY.md 8(d): the same SSG step with BASELINE.json's "(3+6)" wording -- 6 feature channels next to
    xyz (SA1 K = 9, FP4 K = 134) instead of semantic.json's 3; device-resident inputs, graph replay."""
    import torch
    from pn2_b200.train_step import Trainer
    hp = dict(HP, use_color=2)
    rs = np.random.RandomState(100)
    xyz = rs.random_sample((b, n, 3)) * np.array([10.0, 10.0, 5.0]) - np.array([5.0, 5.0, 0.0])
    pc = np.concatenate([xyz, rs.random_sample((b, n, 6))], -1).astype(np.float32)
    labels = rs.randint(1, 9, (b, n)).astype(np.int32)
    smpw = np.ones((b, n), np.float32)
    d = [torch.as_tensor(x).to(dev) for x in (pc, labels, smpw)]
    tr = Trainer(hp, NUM_CLASS, device=dev, seed=0, world_size=1, geometry_ahead=ahead)  # same mode as the headline
    tr.step(*d)
    graph = tr.capture(*d)
    fn = tr.step_graph if graph else tr.step
    for _ in range(max(warmup, 3)):
        fn(*d)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        ev[i][0].record()
        fn(*d)
        ev[i][1].record()
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(bb) for a, bb in ev) / steps
    return {"workload": "ssg_train_step_B%d_N%d_xyz3+feat6 (BASELINE.json wording)" % (b, n),
            "ms_per_step": ms, "value": b * n / (ms * 1e-3), "unit": UNIT, "cuda_graph": bool(graph),
            "geometry_ahead": bool(ahead and graph)}


def fused_chain_bytes(b):
    """The OTHER byte model of the dense stage (VERDICT r1 item 3): if every shared-MLP chain kept its
    intermediates on chip, a chain would read its input X0[M,K0] and write its (pooled) output in the forward,
    and read X0 + the upstream gradient and write dX0 (where an input gradient exists) in the backward."""
    from pn2_b200.model import FP_MLPS, SA_MLPS
    n0 = HP["num_point"]
    npts = [n0, HP["l1_npoint"], HP["l2_npoint"], HP["l3_npoint"], HP["l4_npoint"]]
    feat = [3, 64, 128, 256, 512]
    tot = 0
    for l in (1, 2, 3, 4):
        m = b * npts[l] * HP["l%d_nsample" % l]
        k0, out = feat[l - 1] + 3, b * npts[l] * SA_MLPS[l - 1][-1]
        tot += 4 * (m * k0 + out) + 4 * (m * k0 + out + (m * k0 if l > 1 else 0))
    up = 512
    for l, lo in zip((1, 2, 3, 4), (3, 2, 1, 0)):
        m, k0 = b * npts[lo], up + feat[lo]
        out = m * FP_MLPS[l - 1][-1]
        tot += 4 * (m * k0 + out) + 4 * (2 * m * k0 + out)
        up = FP_MLPS[l - 1][-1]
    m = b * n0
    tot += 4 * (m * 128 + m * NUM_CLASS) + 4 * (2 * m * 128 + m * NUM_CLASS)
    return tot


def step_state(trainer):
    """The tensors a training step reads and updates besides its batch: weights, Adam moments, dropout counter,
    BatchNorm moving statistics."""
    return [trainer.flat, trainer.m, trainer.v, trainer._seed_dev] + trainer._moving()


def dump_outputs(out_dir, trainer, loss):
    """What the last timed step computed, as float32 .npy files: the loss it returned, the gradient it took, the
    weights after its optimizer update and the BatchNorm moving statistics it updated.  Same arguments, same
    seeded inputs, same starting state: two runs or two builds can be compared file by file."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.reshape(1), "grads": trainer.grads, "weights": trainer.flat,
              "bn_moving_stats": torch.cat([t.reshape(-1) for t in trainer._moving()])}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    import pn2_b200
    from pn2_b200 import _ffi
    from pn2_b200.train_step import Trainer
    from pn2_b200.util import tf_util

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        dist.init_process_group("nccl", rank=rank, world_size=world,
                                device_id=torch.device("cuda", local),
                                timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local)
    b, n = args.batch, args.npoint
    # NBATCH distinct synthetic batches, rotated step by step (resident in HBM for `value`, in pinned host memory for
    # `e2e`): every step samples, groups and trains on data the previous step has not seen
    host_batches = [make_batch(b, n, 100 + rank + 1000 * j) for j in range(NBATCH)]
    pc, labels, smpw = host_batches[0]
    dev_batches = [tuple(torch.as_tensor(x).to(dev) for x in hb) for hb in host_batches]
    d_pc, d_lab, d_w = dev_batches[0]
    ahead = not (args.no_ahead or args.no_graph)
    trainer = Trainer(HP, NUM_CLASS, device=dev, seed=0, world_size=world, geometry_ahead=ahead)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Every timed step starts from the freshly initialised model: one pass that updates nothing creates the
    # variables, and their state is put back before each timed step.  A step is deterministic up to the order
    # of its fp32 atomics, but training on compounds that (Adam moves every weight whose gradient is near zero
    # by a whole learning rate, whichever way the rounding tipped its sign), so a timed step that continued
    # the warm-up's training would compute something different in every run.
    with tf_util.frozen_moving_stats():
        trainer.forward_backward(d_pc, d_lab, d_w)
    start_count, start = trainer.step_count, [t.clone() for t in step_state(trainer)]
    trainer.step(d_pc, d_lab, d_w)
    trainer.step(d_pc, d_lab, d_w)
    use_graph = (not args.no_graph) and trainer.capture(d_pc, d_lab, d_w)
    if not use_graph and not args.no_graph:
        print("CUDA-graph capture failed, eager launches instead:\n%s" % trainer._capture_error,
              file=sys.stderr)
    step_fn = trainer.step_graph if use_graph else trainer.step
    launches_per_step = None
    for i in range(max(args.warmup, 3)):
        step_fn(*dev_batches[i % NBATCH])
    barrier()

    # ---- device-resident timing ---------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    calls0 = _ffi.launches
    barrier()
    for i in range(args.steps):
        trainer.step_count = start_count
        torch._foreach_copy_(step_state(trainer), start)
        flush.zero_()
        ev[i][0].record()
        loss = step_fn(*dev_batches[i % NBATCH])
        ev[i][1].record()
    barrier()
    calls = _ffi.launches - calls0
    if use_graph:  # replayed launches are not seen by the ctypes counter: count them from the capture
        calls = args.steps * (trainer.launches_per_replay + 1)
    ms = sum(a.elapsed_time(bb) for a, bb in ev)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, loss)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * b * n * args.steps / (ms_total * 1e-3)

    # ---- end to end: pinned host inputs in, loss out, every step ---------------------------------
    # The public call: Trainer.stage(pinned host batch) starts the H2D copy of the NEXT batch on the copy
    # stream, Trainer.step_graph() consumes it (double-buffered input feed, like the reference's prefetch
    # queue, train.py:134-196).  Every timed step contains exactly one H2D copy of a full batch and one D2H
    # read of the loss; the same 256 MB L2 flush as above runs between steps, outside the events.
    pinned = [tuple(torch.as_tensor(x).pin_memory() for x in hb) for hb in host_batches]
    h_pc, h_lab, h_w = pinned[0]
    h_loss = torch.empty((), dtype=torch.float32).pin_memory()
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(args.steps)]
    barrier()
    last = 0.0
    if use_graph:
        trainer.stage(h_pc, h_lab, h_w)       # fills the pipe (the copy of step 0's batch is timed below
        torch.cuda.synchronize()              # as the copy issued during the last step)
    for i in range(args.steps):
        flush.zero_()
        ev2[i][0].record()
        if use_graph:
            loss = trainer.step_graph()               # consumes the staged batch
            trainer.stage(*pinned[(i + 1) % NBATCH])  # H2D of the next batch overlaps this step
        else:
            loss = trainer.step(*pinned[i % NBATCH])  # eager: H2D on the replica's stream
        h_loss.copy_(loss, non_blocking=True)         # device -> host read of the step's result
        ev2[i][1].record()
        ev2[i][1].synchronize()
        last = float(h_loss)
    barrier()
    t2 = torch.tensor([sum(a.elapsed_time(bb) for a, bb in ev2)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * b * n * args.steps / (float(t2.item()) * 1e-3)
    h2d = int(pc.nbytes + labels.nbytes + smpw.nbytes)

    # ---- per-entry-point breakdown (separate instrumented pass) + roofline ------------------
    roofline, breakdown, collective, linear_table = None, None, None, None
    # every rank takes the instrumented steps (they contain the gradient all-reduce); rank 0 records
    _ffi.profile = [] if rank == 0 else None
    trainer.timing = {}
    torch.cuda.synchronize()
    psteps = min(args.steps, 3)
    side_sms, trainer.wgrad_sms = trainer.wgrad_sms, 0  # every kernel alone on the device: no overlapped streams
    for _ in range(psteps):
        flush.zero_()
        # keep the launch queue backlogged (a ~25 ms spin kernel first): the events around every
        # entry point then time GPU execution only, not the gaps of the eager Python launches
        torch.cuda._sleep(50_000_000)
        trainer.step(d_pc, d_lab, d_w)
    torch.cuda.synchronize()
    trainer.wgrad_sms = side_sms
    barrier()
    if rank == 0:
        agg = {}
        per_shape = {}
        for name, a, bb, shape in _ffi.profile:
            d = agg.setdefault(name, [0.0, 0])
            ms1 = a.elapsed_time(bb)
            d[0] += ms1
            d[1] += 1
            if shape is not None:
                ps = per_shape.setdefault((name,) + tuple(int(x) for x in shape), [0.0, 0])
                ps[0] += ms1
                ps[1] += 1
        _ffi.profile = None
        ar = trainer.timing.get("allreduce", [])
        if ar:
            nbytes = trainer.grads.numel() * 4
            us = 1e3 * sum(a.elapsed_time(bb) for a, bb in ar) / len(ar)
            collective = {"op": "all_reduce(sum) of the flat gradient buffer", "bytes": nbytes,
                          "us_per_step": us,
                          "model_us": 2.0 * (world - 1) / world * nbytes / 900e9 * 1e6,
                          "note": "CUDA events on the replica's stream around dist.all_reduce in the "
                                  "instrumented (eager, backlogged) pass; model = 2(p-1)/p * bytes / 900 GB/s"}
        breakdown = {k: {"ms_per_step": v[0] / psteps, "calls_per_step": v[1] / psteps}
                     for k, v in sorted(agg.items(), key=lambda kv: -kv[1][0])}
        # every GEMM call of a step with its algorithmic bytes 4*M*(K+N) against the measured copy bandwidth
        linear_table = []
        for (name, m_, k_, n_), v in sorted(per_shape.items(), key=lambda kv: -kv[1][0]):
            us = 1e3 * v[0] / v[1]
            byt = 4.0 * m_ * (k_ + n_)
            linear_table.append({"call": name[len("pn2_linear_"):].replace("fwd_bn", "fwd"), "M": m_, "K": k_, "N": n_,
                                 "calls_per_step": v[1] / psteps, "us": us, "GBps": byt / us / 1e3})
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        tc_peak = peaks.get("bf16_tflops_sustained", 1400.0)
        src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        traffic = None
        tf = os.path.join(ROOT, "profiles", "traffic_r02.json")
        if os.path.exists(tf):
            traffic = json.load(open(tf))
        names = ("pn2_linear_fwd", "pn2_linear_dgrad", "pn2_linear_wgrad")
        # the forward of a train-mode BN layer goes through pn2_linear_fwd_bn (GEMM + fused finalize): same kernel
        groups = (("pn2_linear_fwd", "pn2_linear_fwd_bn"), ("pn2_linear_dgrad",), ("pn2_linear_wgrad",))
        lin_ms = [sum(breakdown.get(k, {"ms_per_step": 0.0})["ms_per_step"] for k in g) for g in groups]
        lin_calls = [sum(breakdown.get(k, {"calls_per_step": 0})["calls_per_step"] for k in g) for g in groups]
        lin = sum(lin_ms)
        fps_ms = breakdown.get("pn2_fps", {"ms_per_step": 0.0})["ms_per_step"]
        if fps_ms >= lin:
            byt = sum(fps_stream_bytes(b))
            ach = byt / (fps_ms * 1e-3) / 1e9
            roofline = {"kernel": "pn2_fps (fps_pruned_kernel / fps_reg_kernel, 4 launches/step)", "bound": "hbm",
                        "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                        "traffic": None, "peak_source": src,
                        "model": "streaming-model bytes B*(npoint-1)*N*20 (SURVEY.md 8d); the cloud "
                                 "is register/smem resident so achieved may exceed HBM peak",
                        "us_per_round": fps_ms * 1e3 / sum(m - 1 for m in (1024, 256, 64, 16))}
        else:
            # dominant kernels: tc::tc_gemm_kernel (forward + dgrad) and tcw::tc_wgrad_kernel.  With
            # K, N <= 512 and fp32 activations they are HBM-bound, not tensor-bound.
            byts = gemm_bytes(b)
            ach = sum(byts) / (lin * 1e-3) / 1e9
            fl = 3 * gemm_flops(b)
            roofline = {"kernel": "tc::tc_gemm_kernel + tcw::tc_wgrad_kernel (pn2_linear_fwd/dgrad/wgrad, "
                                  "%d launches/step)" % int(sum(lin_calls)),
                        "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                        "frac": ach / hbm_peak,
                        "traffic": (traffic or {}).get("tcgemm"),
                        "traffic_detail": traffic, "peak_source": src + ", copy bandwidth",
                        "model": "algorithmic bytes 4*M*(K+N) per call (fwd: X in, Y out; dgrad: dY in, dX "
                                 "out; wgrad: X and dY in) over the %.2f ms the three entry points take "
                                 "per step (CUDA events on the launching stream, queue backlogged)" % lin,
                        "per_entry_point": {k: {"ms_per_step": t, "GBps": bb / (t * 1e-3) / 1e9 if t else None}
                                            for k, t, bb in zip(names, lin_ms, byts)},
                        "fused_chain_model": (lambda dense_ms, fb: {
                            "bytes": fb, "dense_stage_ms": dense_ms,
                            "achieved": fb / (dense_ms * 1e-3) / 1e9, "frac": fb / (dense_ms * 1e-3) / 1e9 / hbm_peak,
                            "note": "bytes if every shared-MLP chain kept its intermediates on chip (chain input "
                                    "+ output, + upstream gradient and input gradient in the backward) over the time "
                                    "of the whole dense stage (pn2_linear_*, pn2_bn_*, pn2_affine_act*): the headroom "
                                    "chain fusion would open, next to the per-layer model above"})(
                            sum(v["ms_per_step"] for k, v in breakdown.items()
                                if k.startswith(("pn2_linear_", "pn2_bn_", "pn2_affine_act"))), fused_chain_bytes(b)),
                        "tensor": {"achieved_tflops": fl / (lin * 1e-3) / 1e12,
                                   "peak_tflops_bf16_sustained": tc_peak,
                                   "note": "3xTF32: effective tensor peak is TF32/3 = bf16/6"}}

    # ---- CPU baseline on the host cores (rank 0, N=1 only) ---------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, sec, cores = time_cpu(b, n, 3, 1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "3 steps of the SAME config (%d clouds x %d points, SSG fwd+bwd): C oracle index ops "
                         "(OpenMP over clouds) + PyTorch-CPU fp32 layers, %.2f s/step" % (b, n, sec)}

    cfg1 = cf6 = None
    if rank == 0 and world == 1 and not args.no_extra:
        try:
            cfg1 = config1_row(dev)
        except Exception as e:  # noqa: BLE001
            cfg1 = {"error": repr(e)[:300]}
        try:
            cf6 = cfeat6_line(dev, b, n, min(args.steps, 10), args.warmup, flush, ahead=ahead)
        except Exception as e:  # noqa: BLE001
            cf6 = {"error": repr(e)[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(b, n), "global_batch": b * world,
                       "parallelism": "dp%d" % world, "cuda_graph": bool(use_graph),
                       "wgrad_stream_sms": trainer.wgrad_sms,
                       "batches": "%d distinct synthetic batches rotated step by step (resident in HBM for value, "
                                  "pinned host memory for e2e)" % NBATCH,
                       "start_state": "every step of value starts from the freshly initialised model "
                                      "(restored outside the events)",
                       "geometry_ahead": ("every replay = dense stage of the current batch + sampling / neighbour "
                                          "search of the next batch on a second stream of the same graph; K steps "
                                          "run K of each") if (ahead and use_graph) else False,
                       "cuda_graph_error": (trainer._capture_error or "")[:1500] or None,
                       "l2": "256 MB flush write between timed steps; a step also streams >1 GB of "
                             "activations, far beyond the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "last_loss": last,
                    "feed": "Trainer.stage(pinned host batch) + Trainer.step_graph(): one H2D batch copy and one "
                            "D2H loss read per step, the copy of batch i+1 overlaps step i" +
                            ("; geometry-ahead: the batch copied in during step i is sampled / grouped by step i+1's "
                             "replay and trained on by step i+2's, the loss read is that of the batch trained on"
                             if (ahead and use_graph) else "")},
            "gpu_launches": calls,
            "roofline": roofline, "cpu_baseline": cpu, "breakdown_ms_per_step": breakdown,
            "collective": collective, "config1": cfg1, "cfeat6": cf6, "linear_calls": linear_table,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="clouds per GPU")
    ap.add_argument("--npoint", type=int, default=8192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of a CUDA graph")
    ap.add_argument("--no-ahead", action="store_true",
                    help="compute the geometry (FPS, ball query, 3-NN) of a batch inside its own step instead of "
                         "one batch ahead on a second stream")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the config-1 row and the 6-feature-channel line (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the engine's timed step computed: --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
