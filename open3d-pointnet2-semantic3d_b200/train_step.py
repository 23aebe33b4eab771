"""One training step of the reference's train.py on the sm_100a engine.

  get_learning_rate / get_bn_decay                       train.py:80-119
  Trainer.step: forward, loss, backward, Adam            train.py:387-388, 225-244
  data parallelism: batch sharded across ranks, ONE NCCL all-reduce over the flat gradient
  buffer per step (SURVEY.md section 8e); BatchNorm statistics stay per replica.
  Trainer.evaluate: eval-mode forward + loss + confusion      train.py:263-330 (sess.run([loss, pred]), :296-312)
  Trainer.train_confusion: confusion of every training pass  train.py:234-251

Stream discipline: a Trainer owns ONE CUDA stream and issues every launch of its replica on it --
the eager passes, the CUDA-graph capture and the replays alike.  The autograd engine ties each
backward node (and the accumulation of leaf gradients) to the stream its forward ran on; mixing
the default stream (eager warm-up) with a capture stream made the engine create a dependency on
uncaptured work (cudaErrorStreamCaptureIsolation) at the end of the captured backward, which is
how graph mode silently fell back to eager launches in round 1.  The caller's current stream is
joined at the start and at the end of every step, so callers keep ordinary stream semantics.
Two side streams branch off it and are joined again inside every pass (and inside the captured graph): the
weight gradients of the backward pass (util/tf_util.py, set_wgrad_stream: dW = A^T dY of a layer is independent
of the input-gradient / BatchNorm-backward chain once dY exists, so the tensor-core wgrad runs on 64 SMs next
to the HBM-bound BatchNorm kernels instead of after them), and, in geometry_ahead mode, the geometry stream.

Geometry one batch ahead (``Trainer(..., geometry_ahead=True)``, graph mode): farthest point sampling,
gather, ball query, 3-NN and the interpolation weights depend on the coordinates only, yet they head the
critical path of a step (~0.9 of ~4.1 ms at B=16 x 8192; FPS alone keeps 16 of 148 SMs busy for 0.5 ms while
132 idle).  In this mode one replay runs the dense stage (grouping, shared MLPs, loss, backward) of the
CURRENT batch from a precomputed GeometryTape and, forked onto a second stream inside the same graph, the
geometry of the NEXT batch; the persistent tensor-core GEMMs of the forward pass size their grids for the SMs
the sampling kernels leave free (pn2_set_sm_budget).  The reference overlaps its host-side batch preparation
with training the same way (train.py:134-196).  Nothing is cached or skipped: K replays run K dense stages and
K geometry stages, on the same kernels, and the values the dense stage consumes are the ones the plain step
computes (tests/test_train_step_gpu.py compares the two step by step).
"""
import gc
import os

import torch
import torch.distributed as dist

from . import _ffi, model
from ._ffi import F32, call, ptr
from .util import pointnet_util, tf_util
from .util.metric import ConfusionMatrix


def get_learning_rate(step, params):
    """tf.train.exponential_decay(staircase) clipped at 1e-5 (train.py:80-97)."""
    lr = params["learning_rate"] * params["learning_rate_decay_rate"] ** (
        (step * params["batch_size"]) // params["decay_step"])
    return max(lr, 0.00001)


def get_bn_decay(step, params):
    """min(clip, 1 - init*rate^floor(step*B/decay_step)) (train.py:100-119)."""
    mom = params["bn_init_decay"] * params["bn_decay_decay_rate"] ** (
        (step * params["batch_size"]) // int(params["decay_step"]))
    return min(params["bn_decay_clip"], 1 - mom)


def shard_batch(global_batch, rank, world_size):
    """Contiguous shard of the leading (cloud) dimension owned by ``rank``: the path is
    independent per cloud, so data parallelism partitions clouds with no data-path exchange."""
    total = global_batch.shape[0]
    if world_size < 1 or not 0 <= rank < world_size or total % world_size != 0:
        raise ValueError("cannot shard %d clouds over %d ranks (rank %d): the batch must divide evenly"
                         % (total, world_size, rank))
    per = total // world_size
    return global_batch[rank * per:(rank + 1) * per]


def allreduce_flat(flat_grads, world_size):
    """The single collective of a step: SUM all-reduce of the flat gradient buffer.  Returns the
    scale (1/world_size) the Adam kernel folds into its gradient read."""
    if world_size > 1:
        dist.all_reduce(flat_grads, op=dist.ReduceOp.SUM)
    return 1.0 / world_size


class Trainer:
    """Owns the variables, Adam moments, step counter and the CUDA stream of one replica.

    Dropout: the mask of step k (1-based) is drawn with seed ``host_seed + k`` -- a device-resident
    counter that every step increments, in eager and in graph mode alike, so a replayed graph sees
    a fresh mask and both modes walk through the same mask sequence.
    """

    def __init__(self, params, num_class, device="cuda", seed=0, world_size=1, geometry_ahead=False,
                 wgrad_sms=None):
        self.params, self.num_class, self.world_size = params, num_class, world_size
        self.geometry_ahead = bool(geometry_ahead)
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.store = tf_util.set_default_store(tf_util.VariableStore(device=self.device, seed=seed))
        self.step_count = 0
        self.flat = self.grads = self.m = self.v = None
        self.stream = torch.cuda.Stream(device=self.device)
        self._copy_stream = torch.cuda.Stream(device=self.device)
        self._seed_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._graph = None
        self._static = self._staging = None
        self._staged_event = self._consumed_event = None
        self._capture_error = None
        self.launches_per_replay = 0
        self.timing = None  # bench.py: dict that receives CUDA events around the collective
        # geometry one batch ahead: the tape the dense stage of the current batch consumes, the inputs of the
        # batch whose geometry is computed meanwhile, the stream that computes it
        self._tape = self._next = None
        # SMs the forward GEMMs leave free in a pass WITHOUT a geometry stream (0 = none).  A test hook: the fp32
        # partial sums of the BatchNorm statistics depend on which tiles a CTA owns, i.e. on the grid size, so a
        # single-stream reference for the geometry-ahead mode has to run its forward GEMMs on the same grid
        self.forward_reserve = 0
        # SMs the weight-gradient GEMMs get on their own stream during the backward pass (0 = same stream as the
        # rest).  64 of 148 measured best at B=16 x 8192 (3.52 -> 3.30 ms per step; 48: 3.35, 80: 3.36, a stream
        # priority for the main chain changed nothing)
        self.wgrad_sms = int(os.environ.get("PN2_WGRAD_SMS", "64")) if wgrad_sms is None else int(wgrad_sms)
        self._wstream = torch.cuda.Stream(device=self.device) if self.wgrad_sms > 0 else None
        self._side = torch.cuda.Stream(device=self.device) if self.geometry_ahead else None
        # a util.metric.ConfusionMatrix: every training pass adds the confusion of its training-mode logits
        # (dropout applied, the train op's `pred` of train.py:234-251); part of the captured step graph, so setting
        # or clearing it re-captures on the next step_graph
        self.train_confusion = None
        self._graph_train_confusion = None
        # evaluate(): one graph per batch shape (None = eager, the reason in _eval_capture_error); the pass counts
        # into a trainer-owned matrix that the graph zeroes, so the caller's matrix is not baked into the graph
        self._eval_graphs = {}
        self._eval_cm = None
        self._eval_capture_error = None

    # ---- variables ----------------------------------------------------------------------------
    def _ensure_flat(self):
        if self.store.flat_params is None:
            self.flat, self.grads = self.store.flatten()
            self.m = torch.zeros_like(self.flat)
            self.v = torch.zeros_like(self.flat)
            self.store.allocate_images()
            if self.world_size > 1:  # replicas start from rank 0's weights
                dist.broadcast(self.flat, src=0)

    def _moving(self):
        return [v.data for v in self.store.vars.values() if not v.trainable]

    # ---- one forward + loss + backward on self.stream --------------------------------------------
    def _fb(self, point_cloud, labels, smpw, ahead=None):
        """``ahead`` = (point_cloud, labels, smpw) of the NEXT batch: the dense stage of this pass takes its
        geometry from self._tape while the geometry of the next batch is computed on the side stream; at the
        end the tape and the current inputs are overwritten with the next batch's."""
        bn_decay = get_bn_decay(self.step_count, self.params)
        tf_util.set_default_store(self.store)
        tf_util.set_dropout_seed_device(self._seed_dev)
        # a fresh autograd anchor per pass: no leaf (or its gradient accumulator) outlives the pass
        self.store.anchor = torch.zeros(1, device=self.device, requires_grad=True)
        tf_util.zero_arena.reset(self.device)  # one memset for every layer's fp64 accumulators
        if self._wstream is not None and os.environ.get("PN2_PREP_SIDE", "1") != "0":
            # one launch: every layer's 3xTF32 weight images -- on the side stream, the first GEMM waits for it
            # (the main stream meanwhile gathers and centres SA1's groups)
            self._wstream.wait_stream(self.stream)
            with torch.cuda.stream(self._wstream):
                self.store.prepare_images()
                ev = torch.cuda.Event()
                ev.record(self._wstream)
            tf_util.set_images_event(ev)
        else:
            self.store.prepare_images()
        nxt = None
        if ahead is not None:
            self._side.wait_stream(self.stream)  # fork
            with torch.cuda.stream(self._side):
                nxt = model.get_geometry(ahead[0], self.params)
        try:
            with pointnet_util.replay_geometry(self._tape if ahead is not None else None):
                self._sm_budget(point_cloud.shape[0] if ahead is not None else self.forward_reserve)
                try:
                    pred, _ = model.get_model(point_cloud, True, self.num_class, self.params, bn_decay=bn_decay)
                finally:
                    if os.environ.get("PN2_AHEAD_SCOPE", "fwd") != "step":
                        self._sm_budget(0)
                if self.train_confusion is not None:
                    self.train_confusion.increment_from_logits(pred.detach(), labels.to(torch.int32).contiguous())
                self.store.zero_grad()
                loss = model.get_loss(pred, labels, smpw)
                if self.wgrad_sms > 0:  # weight gradients next to the rest of the backward pass (util/tf_util.py)
                    tf_util.set_wgrad_stream(self._wstream, self.wgrad_sms)
                try:
                    loss.backward()
                finally:
                    if self.wgrad_sms > 0:
                        tf_util.set_wgrad_stream(None)
                        _ffi.lib().pn2_set_sm_budget(0)
                        self.stream.wait_stream(self._wstream)  # join: every weight gradient is complete
        finally:
            self._sm_budget(0)
            tf_util.set_images_event(None)
            tf_util.zero_arena.disarm()
            tf_util.set_dropout_seed_device(None)
            self.store.images_fresh = False  # the optimizer step that follows changes the weights
        if ahead is not None:
            self.stream.wait_stream(self._side)  # join: the dense stage has read its tape, the next one is complete
            torch._foreach_copy_(self._tape.tensors(), nxt.tensors())
            torch._foreach_copy_([point_cloud, labels, smpw], list(ahead))
            if not torch.cuda.is_current_stream_capturing():
                for t in nxt.tensors():
                    t.record_stream(self.stream)  # allocated on the side stream, last read on this one
        return loss.detach()

    def _sm_budget(self, reserve):
        """Leave ``reserve`` SMs (one per cloud: the FPS kernel runs one CTA per cloud) to the geometry stream."""
        if not self.geometry_ahead and not self.forward_reserve:
            return
        if reserve:
            reserve = int(os.environ.get("PN2_AHEAD_RESERVE", min(int(reserve), 32)))
        total = torch.cuda.get_device_properties(self.device).multi_processor_count
        _ffi.lib().pn2_set_sm_budget(total - reserve if 0 < reserve < total else 0)

    def _create_variables(self, point_cloud):
        """The first forward pass creates the variables (the reference builds its graph once,
        model.py:22-148); it runs with BatchNorm's moving statistics frozen and its result is
        discarded, so step 1 applies exactly one EMA update like the reference's first train op."""
        if self.store.flat_params is not None:
            return
        tf_util.set_default_store(self.store)
        tf_util.set_dropout_seed_device(self._seed_dev)
        tf_util.zero_arena.reset(self.device)
        try:
            with torch.no_grad(), tf_util.frozen_moving_stats():
                model.get_model(point_cloud, True, self.num_class, self.params,
                                bn_decay=get_bn_decay(self.step_count, self.params))
        finally:
            tf_util.zero_arena.disarm()
            tf_util.set_dropout_seed_device(None)
        self._ensure_flat()

    def forward_backward(self, point_cloud, labels, smpw):
        """Forward + loss + backward (gradients land in the flat gradient buffer); no optimizer
        step, the dropout counter is not advanced."""
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            point_cloud, labels, smpw = self._to_device(point_cloud, labels, smpw)
            self._create_variables(point_cloud)
            loss = self._fb(point_cloud, labels, smpw)
        caller.wait_stream(self.stream)
        return loss

    def _to_device(self, *ts):
        return tuple(t if t.is_cuda else t.to(self.device, non_blocking=True) for t in ts)

    # ---- eager step ------------------------------------------------------------------------------
    def step(self, point_cloud, labels, smpw):
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            point_cloud, labels, smpw = self._to_device(point_cloud, labels, smpw)
            self._create_variables(point_cloud)
            self._seed_dev.add_(1)
            loss = self._fb(point_cloud, labels, smpw)
            self._apply_gradients()
        caller.wait_stream(self.stream)
        return loss

    def _apply_gradients(self):
        ev = None
        if self.timing is not None and self.world_size > 1:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        gscale = allreduce_flat(self.grads, self.world_size)
        if ev is not None:
            ev[1].record()
            self.timing.setdefault("allreduce", []).append(ev)
        self.step_count += 1
        lr = get_learning_rate(self.step_count - 1, self.params)
        call("pn2_adam_step", self.flat.numel(), ptr(self.flat, F32), ptr(self.grads, F32),
             ptr(self.m, F32), ptr(self.v, F32), float(lr), 0.9, 0.999, 1e-8, self.step_count,
             float(gscale))

    # ---- CUDA-graph mode: forward + loss + backward captured once, replayed per step -------------
    def capture(self, point_cloud, labels, smpw):
        """Capture forward+loss+backward of this batch shape into a CUDA graph (the ~190 entry-point
        calls of a step are otherwise CPU-launch bound).  Schedule values that are baked in
        (bn_decay) trigger a re-capture when they change.  The warm-up passes and the validation
        replay leave no trace: moving statistics are frozen / restored, the dropout counter is not
        advanced, no optimizer step is taken.  Returns False (eager mode stays) if capture fails;
        the reason is kept, untruncated, in ``self._capture_error``.  In geometry_ahead mode the graph is
        captured around the batch loaded by ``prime()`` (the arguments prime the pipeline if it is empty and are
        otherwise ignored): the pipeline state survives a re-capture."""
        self._graph = None
        self._capture_error = None
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        try:
            with torch.cuda.stream(self.stream):
                src = self._to_device(point_cloud, labels, smpw)
                self._create_variables(src[0])
                ahead = None
                if self.geometry_ahead:
                    # the pipeline state survives a (re-)capture: with next = current, the warm-up passes and
                    # the validation replay recompute the tape of the current batch and copy the batch onto itself
                    if self._tape is None:
                        self._prime(src)
                    for d, s in zip(self._next, self._static):
                        d.copy_(s)
                    ahead = self._next
                elif self._static is None or any(a.shape != b.shape for a, b in zip(self._static, src)):
                    self._static = [t.clone() for t in src]
                else:
                    for d, s in zip(self._static, src):
                        if d.data_ptr() != s.data_ptr():
                            d.copy_(s)
                static = self._static
                # the warm-up passes and the validation replay count too: their counts are undone below
                cm = self.train_confusion
                keep_cm = None if cm is None else cm._counts.clone()
                with tf_util.frozen_moving_stats():
                    for _ in range(2):  # every kernel / workspace / gradient buffer exists
                        self._fb(*static, ahead=ahead)
                self.stream.synchronize()
                for st in (self._side, self._wstream):
                    if st is not None:
                        st.synchronize()
                gc.collect()  # no autograd graph of an earlier pass survives into the capture
                g = torch.cuda.CUDAGraph()
                n0 = _ffi.launches
                with torch.cuda.graph(g, stream=self.stream, capture_error_mode="thread_local"):
                    loss = self._fb(*static, ahead=ahead)
                self.launches_per_replay = _ffi.launches - n0
                # validation replay (would raise on a broken graph), then undo its EMA update
                keep = [t.clone() for t in self._moving()]
                g.replay()
                self.stream.synchronize()
                for t, k in zip(self._moving(), keep):
                    t.copy_(k)
                if cm is not None:
                    cm._counts.copy_(keep_cm)
                self._static_loss = loss
                self._graph = g
                self._graph_bn_decay = get_bn_decay(self.step_count, self.params)
                self._graph_train_confusion = cm
        except Exception as e:  # noqa: BLE001 - any capture failure means eager mode
            import traceback
            self._graph = None
            self._capture_error = repr(e) + " | " + traceback.format_exc()
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
        caller.wait_stream(self.stream)
        return self._graph is not None

    # ---- geometry one batch ahead -----------------------------------------------------------------------
    def _prime(self, src):
        self._static = [t.clone() for t in src]
        self._next = [t.clone() for t in src]
        self._tape = model.get_geometry(self._static[0], self.params)

    def prime(self, point_cloud, labels, smpw):
        """geometry_ahead mode: load the FIRST batch (its geometry is computed here, on the replica's stream).
        Every ``step_graph(batch)`` after that trains on the batch loaded before it and returns that batch's
        loss, while the geometry of ``batch`` is computed alongside."""
        if not self.geometry_ahead:
            raise ValueError("prime() belongs to Trainer(..., geometry_ahead=True)")
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            src = self._to_device(point_cloud, labels, smpw)
            self._create_variables(src[0])
            if self._tape is None or any(a.shape != b.shape for a, b in zip(self._static, src)):
                self._prime(src)
                self._graph = None
            else:
                for d, s in zip(self._static, src):
                    d.copy_(s)
                torch._foreach_copy_(self._tape.tensors(), model.get_geometry(self._static[0], self.params).tensors())
        caller.wait_stream(self.stream)

    def stage(self, point_cloud, labels, smpw):
        """Start the host->device copy of the NEXT batch on the copy stream (pinned host tensors);
        ``step_graph()`` without arguments consumes it.  This is the double-buffered input feed
        (the reference prefetches batches with a process pool, train.py:134-196)."""
        src = (point_cloud, labels, smpw)
        if self._staging is None or any(a.shape != b.shape for a, b in zip(self._staging, src)):
            self._staging = [torch.empty(t.shape, dtype=t.dtype, device=self.device) for t in src]
        cs = self._copy_stream
        cs.wait_stream(torch.cuda.current_stream(self.device))
        if self._consumed_event is not None:
            cs.wait_event(self._consumed_event)  # the previous staged batch has been copied out
        with torch.cuda.stream(cs):
            for d, s in zip(self._staging, src):
                d.copy_(s, non_blocking=True)
            self._staged_event = torch.cuda.Event()
            self._staged_event.record(cs)

    def step_graph(self, point_cloud=None, labels=None, smpw=None):
        """One step by graph replay.  Inputs: device tensors, pinned host tensors (copied in on the
        replica's stream), or nothing at all = the batch handed to ``stage()``.  In geometry_ahead mode the
        inputs are the NEXT batch (see ``prime``); the loss returned is that of the batch trained on."""
        staged = point_cloud is None
        if staged:
            if self._staged_event is None:
                raise ValueError("step_graph() without inputs needs a batch from stage()")
            src = self._staging
        else:
            src = (point_cloud, labels, smpw)
        if self.geometry_ahead:
            # the batch handed in is the one whose geometry this replay computes; the dense stage trains on the
            # batch of the previous call (prime() loaded the first one)
            if self._tape is None:
                raise ValueError("geometry_ahead: call prime(first_batch) before the first step_graph(next_batch)")
            if any(a.shape != b.shape for a, b in zip(self._static, src)):
                raise ValueError("geometry_ahead needs a fixed batch shape")
            if self._graph is None or get_bn_decay(self.step_count, self.params) != self._graph_bn_decay or \
                    self.train_confusion is not self._graph_train_confusion:
                if not self.capture(*self._static):
                    raise _ffi.Pn2Error("geometry_ahead needs graph mode; capture failed: %s" % self._capture_error)
            inputs = self._next
        else:
            if self._graph is None:
                if staged:
                    torch.cuda.current_stream(self.device).wait_event(self._staged_event)
                return self.step(*src)
            if get_bn_decay(self.step_count, self.params) != self._graph_bn_decay or \
                    self.train_confusion is not self._graph_train_confusion or \
                    any(a.shape != b.shape for a, b in zip(self._static, src)):
                if staged:
                    torch.cuda.current_stream(self.device).wait_event(self._staged_event)
                if not self.capture(*src):
                    return self.step(*src)
            inputs = self._static
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            if staged:
                self.stream.wait_event(self._staged_event)
            for dst, s in zip(inputs, src):
                if dst.data_ptr() != s.data_ptr():
                    dst.copy_(s, non_blocking=True)
            if staged:
                self._consumed_event = torch.cuda.Event()
                self._consumed_event.record(self.stream)
                self._staged_event = None
            self._seed_dev.add_(1)
            self._graph.replay()
            self._apply_gradients()
        caller.wait_stream(self.stream)
        return self._static_loss

    # ---- evaluation: eval_one_epoch's sess.run([loss, pred]) (train.py:296-312) -------------------------
    def _eval_pass(self, point_cloud, labels, smpw):
        """Eval-mode forward (moving-average BatchNorm, no dropout) + loss, no backward; the confusion of the
        logits goes to self._eval_cm, which the pass zeroes first.  Geometry is computed inline: a geometry-ahead
        tape is neither read nor advanced.  Weights, moving statistics and the dropout counter are only read."""
        tf_util.set_default_store(self.store)
        tf_util.zero_arena.reset(self.device)
        fresh = self.store.images_fresh
        try:
            self.store.prepare_images()  # the weights change between calls: part of the pass (and of its graph)
            with torch.no_grad(), pointnet_util.replay_geometry(None):
                pred, _ = model.get_model(point_cloud, False, self.num_class, self.params)
                loss = model.get_loss(pred, labels, smpw)
                self._eval_cm.reset()
                self._eval_cm.increment_from_logits(pred.contiguous(), labels.to(torch.int32).contiguous())
        finally:
            tf_util.zero_arena.disarm()
            self.store.images_fresh = fresh
        return loss

    def _capture_eval(self, src):
        """-> (graph, static inputs, static loss) of the eval pass for this batch shape, or None (eager mode;
        the reason is kept in self._eval_capture_error)."""
        static = [t.clone() for t in src]
        try:
            self._eval_pass(*static)  # every kernel attribute / buffer exists before the capture
            self.stream.synchronize()
            gc.collect()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream, capture_error_mode="thread_local"):
                loss = self._eval_pass(*static)
            g.replay()  # validation replay (raises on a broken graph); the pass has no side effect to undo
            self.stream.synchronize()
            return g, static, loss
        except Exception as e:  # noqa: BLE001 - any capture failure means eager mode
            import traceback
            self._eval_capture_error = repr(e) + " | " + traceback.format_exc()
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
            return None

    def evaluate(self, point_cloud, labels, smpw, confusion=None, graph=True):
        """Eval-mode loss of one batch (0-dim CUDA tensor, this call's own); with ``confusion`` (a
        util.metric.ConfusionMatrix) the confusion of the eval logits is added to it.  Runs on the replica's
        stream, by replay of a graph captured once per batch shape (``graph=False``: eager launches).  Leaves
        every piece of training state as it was: weights, Adam moments, moving statistics, step and dropout
        counters, the training graph and the geometry-ahead pipeline."""
        if confusion is not None and confusion.num_classes != self.num_class:
            raise ValueError("confusion has %d classes, the model %d" % (confusion.num_classes, self.num_class))
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            src = self._to_device(point_cloud, labels, smpw)
            self._create_variables(src[0])
            if self._eval_cm is None:
                self._eval_cm = ConfusionMatrix(self.num_class, device=self.device)
            entry = None
            if graph:
                key = tuple((tuple(t.shape), t.dtype) for t in src)
                if key not in self._eval_graphs:
                    self._eval_graphs[key] = self._capture_eval(src)
                entry = self._eval_graphs[key]
            if entry is not None:
                g, static, static_loss = entry
                for d, s in zip(static, src):
                    d.copy_(s, non_blocking=True)
                g.replay()
                loss = static_loss.clone()  # the next replay overwrites static_loss
            else:
                loss = self._eval_pass(*src)
            if confusion is not None:
                confusion._counts.add_(self._eval_cm._counts)
        loss.record_stream(caller)
        caller.wait_stream(self.stream)
        return loss
