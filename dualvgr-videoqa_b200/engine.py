"""Data-parallel train step for DualVGR on B200: the loop body of the reference's train.py:131-160 with the device
work restated B200-first.

  * one process per GPU; parameters live in ONE flat fp32 buffer, gradients in another (views handed to autograd), so the
    gradient exchange is a single NCCL all-reduce over NVLink and the optimizer is two kernel launches
  * loss = CE + alpha * mean_l common_loss + beta * mean_l (HSIC_app + HSIC_mot)  (train.py:146-154): the cross-entropy kernel
    produces value and gradient in one launch; the auxiliary terms of every unit layer (values and all four gradients) are
    computed inside the unit stack's autograd Function on a side stream, overlapped with the rest of the step
  * clip_grad_norm_(12) + Adam(lr)  (train.py:85,158-159) = dvgr_sumsq + dvgr_adam_step on the flat buffers

Videos are independent, so ranks shard the batch and never exchange activations. Two cross-sample couplings remain
(SURVEY.md §8e): BatchNorm1d in the classifier uses per-rank batch statistics by default (standard DDP) or global ones with
sync_bn=True (two 2 x 768-float all-reduces per step); CE / common_loss are means (gradient averaging reproduces the
global-batch gradient), HSIC is a SUM over the batch, so its coefficient is multiplied by world_size before averaging."""
import contextlib
import os
import weakref

import torch
import torch.distributed as dist

from . import autograd as ag
from . import fused_stack as fs
from . import ops
from .loader import DeviceFeatureStore

_LIVE_ENGINES = weakref.WeakSet()


class _EarlyBucketHook:
    """Tensor hook shared by the unit stack's inputs (model/models.py: app, mot, dynamic_q, words): when the last of their
    gradients has been produced, every parameter gradient of the early bucket is final -> start its all-reduce on a side
    stream (captured into the step's CUDA graph as a fork; TrainEngine.optimizer_step joins it)."""

    def __init__(self, engine):
        self.engine = engine
        # high priority: the collective's few CTAs must get their SMs BEFORE the encoders' persistent backward kernels fill the
        # GPU (those claim their tiles dynamically, so they simply run on the SMs that are left)
        self.side = torch.cuda.Stream(priority=-1)
        self.pending = 0
        self.fired = False

    def arm(self, n):
        self.pending = n
        self.fired = False

    def __call__(self, grad):
        self.pending -= 1
        if self.pending == 0 and not self.engine.skip_allreduce:
            e = self.engine
            ev = fs.LAST_QUERY_CHAIN_BWD[0]
            if ev is not None:       # the question side of the unit stack ran its backward on the question stream
                torch.cuda.current_stream().wait_event(ev)
            ops.flush_wgrads()       # the queued (deferred) weight gradients of the early bucket must land before it is reduced
            self.side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.side):
                dist.all_reduce(e.gflat[e.late_numel:], op=dist.ReduceOp.SUM, group=e.pg)
            self.fired = True
        return None


class TrainEngine:
    def __init__(self, model, lr=1e-4, max_norm=12.0, alpha=1.0, beta=1e-8, betas=(0.9, 0.999), eps=1e-8,
                 process_group=None, sync_bn=False):
        self.model = model
        self.lr, self.max_norm, self.alpha, self.beta, self.betas, self.eps = lr, max_norm, alpha, beta, betas, eps
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(process_group) if self.world > 1 else 0
        self.skip_allreduce = False      # measurement aid (bench.py: exposed all-reduce time = step with - step without)
        # flat layout: the groups the fused kernels see as one matrix (contiguous, in order) and everything else, split in
        # two contiguous buckets by WHEN the gradient is final: "late" = the three input encoders (their backward runs last:
        # LSTM recurrences + the big W_ih weight gradients, ~2 ms), "early" = everything downstream of them. With more than
        # one rank the early bucket is all-reduced on a side stream while the encoders' backward still runs.
        late_ids = set()
        for name in ("visual_appearance_input_unit", "linguistic_input_unit", "visual_motion_input_unit"):
            m = getattr(model, name, None)
            if m is not None:
                late_ids.update(id(p) for p in m.parameters())
        grouped, seen = [], set()
        for grp in ag.grad_groups(model):
            for p in grp:
                if p.requires_grad and id(p) not in seen:
                    grouped.append(p); seen.add(id(p))
        rest = [p for p in model.parameters() if p.requires_grad and id(p) not in seen]
        late = [p for p in grouped if id(p) in late_ids] + [p for p in rest if id(p) in late_ids]
        early = [p for p in grouped if id(p) not in late_ids] + [p for p in rest if id(p) not in late_ids]
        self.params = late + early
        self._n_late = len(late)
        dev = self.params[0].device
        self.sizes = [(p.numel() + 7) // 8 * 8 for p in self.params]      # 16-byte aligned slices (also in the bf16 shadow)
        total = sum(self.sizes)
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.gflat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.shadow = torch.zeros(total, dtype=torch.bfloat16, device=dev)   # bf16 GEMM operands, written by the Adam kernel
        self.m = torch.zeros(total, dtype=torch.float32, device=dev)
        self.v = torch.zeros(total, dtype=torch.float32, device=dev)
        self.late_numel = sum(self.sizes[:self._n_late])
        off = 0
        with torch.no_grad():
            for p, n in zip(self.params, self.sizes):
                sl = self.flat[off:off + p.numel()].view_as(p)
                sl.copy_(p.data)
                p.data = sl
                p.grad = self.gflat[off:off + p.numel()].view_as(p)
                if p.dim() == 2:
                    ag.SHADOW[id(p)] = (weakref.ref(p), self.shadow[off:off + p.numel()].view_as(p))
                off += n
        self.step_count = 0
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=dev)     # device-side step counter (graph replay)
        self.seed_dev = torch.zeros(1, dtype=torch.int64, device=dev)     # device-side dropout seed offset
        self.graph = None
        self.static = None
        self.numel = total
        # ONE high-priority stream for every step of this engine, eager or captured: kernel nodes inherit the priority of the
        # stream they are recorded on (the critical path must win SMs over the low-priority auxiliary-loss stream), and
        # autograd remembers the stream a parameter was first used on — eager steps on the caller's stream followed by a
        # capture on another one made the captured backward wait on uncaptured work
        self.stream = torch.cuda.Stream(device=dev, priority=-1) if dev.type == "cuda" else None   # (CPU: layout inspection only)
        self.last_stats = None           # [4] f32 device tensor of the last step: total, common sum, dependence sum, #timeouts
        self._step_flags = []
        if self.world > 1:      # replicas must start identical (the reference seeds every process the same, train.py:425-428)
            dist.broadcast(self.flat, src=0, group=self.pg)
        self.sync_shadow()      # AFTER the broadcast: the bf16 operands must be casts of the weights this rank trains on
        # independent dropout masks per rank (standard DDP): the counter-based streams are keyed by (seed, site, element), so
        # the rank goes into the seed; weights were identical before this point
        ag.set_rank_seed(self.rank)
        ag.DIRECT_GRAD[0] = True      # weight-gradient GEMMs accumulate straight into the flat gradient buffer
        # SMs the appearance encoder's backward RECURRENCE leaves to the question encoder's (32 tiles per step: 32 SMs). It is
        # HBM-bound and loses nothing on 116 CTAs, while the question chain behind it no longer queues for SMs (-0.05 ms; the
        # tensor-bound weight-gradient launches are NOT capped: measured slower, DVGR_RESERVE_WGRAD=1 to repeat)
        # default: one SM per tile of a question-encoder step (4 directions x ceil(B / 32) row blocks), at most 64 — measured:
        # SVQA (B=256) 32: -0.05 ms; MSVD (B=1024) 32: +0.14 ms, 64: neutral; 64-clip videos (B=512) 32: -0.5 ms
        self._reserve_env = os.environ.get("DVGR_RESERVE_SMS")
        ops.RESERVE_SMS[0] = int(self._reserve_env) if self._reserve_env is not None else 32
        _LIVE_ENGINES.add(self)
        overlap_ok = os.environ.get("DVGR_ALLREDUCE_OVERLAP", "1") != "0"        # A/B knob: 0 = one all-reduce after backward
        self._overlap = _EarlyBucketHook(self) if (self.world > 1 and overlap_ok and 0 < self.late_numel < total) else None
        if hasattr(model, "_unit_inputs_grad_hook") or self._overlap is not None:
            model._unit_inputs_grad_hook = self._overlap
        self.sync_bn = bool(sync_bn) and self.world > 1
        ou = getattr(model, "output_unit", None)
        if ou is not None:
            ou.sync_bn_group = (self.pg if self.pg is not None else dist.group.WORLD) if self.sync_bn else None
            ou.sync_bn_world = self.world if self.sync_bn else 1

    # ------------------------------------------------------------------------------------------------------------
    def sync_shadow(self):
        """Re-casts the bf16 operand copy from the fp32 master weights. Call after ANY external write to the parameters
        (load_state_dict, manual edits, a restore): the GEMMs read the shadow, not the fp32 values."""
        with torch.no_grad():
            self.shadow.copy_(self.flat)
        ag.invalidate_weight_cache()

    def state_dict(self):
        """Optimizer / engine state for checkpoints (the reference saves optimizer.state_dict(), train.py:359-367): Adam
        moments per parameter NAME (views, compatible with torch.optim.Adam's exp_avg / exp_avg_sq), step, dropout counter."""
        names = {id(p): n for n, p in self.model.named_parameters()}
        st, off = {}, 0
        for p, n in zip(self.params, self.sizes):
            st[names[id(p)]] = {"exp_avg": self.m[off:off + p.numel()].view_as(p).clone(),
                                "exp_avg_sq": self.v[off:off + p.numel()].view_as(p).clone()}
            off += n
        return {"state": st, "step": int(self.step_dev.item()), "seed_offset": int(self.seed_dev.item()),
                "lr": self.lr, "betas": self.betas, "eps": self.eps, "max_norm": self.max_norm}

    def load_state_dict(self, sd):
        names = {id(p): n for n, p in self.model.named_parameters()}
        off = 0
        with torch.no_grad():
            for p, n in zip(self.params, self.sizes):
                ent = sd["state"][names[id(p)]]
                self.m[off:off + p.numel()].view_as(p).copy_(ent["exp_avg"])
                self.v[off:off + p.numel()].view_as(p).copy_(ent["exp_avg_sq"])
                off += n
            self.step_dev.fill_(int(sd["step"]))
            self.seed_dev.fill_(int(sd.get("seed_offset", 0)))
        self.step_count = int(sd["step"])
        self.lr = sd.get("lr", self.lr)
        self.sync_shadow()       # model.load_state_dict() normally precedes this call: pick the restored weights up

    # ------------------------------------------------------------------------------------------------------------
    def _loss_coefs(self, B, N, n_layers):
        n = max(n_layers, 1)
        return (self.alpha / n) / (B * N * N), self.beta * self.world / n

    @contextlib.contextmanager
    def _on_stream(self):
        """Runs the body on the engine's stream, ordered after the caller's current stream and joined back to it."""
        cur = torch.cuda.current_stream()
        if cur == self.stream:
            yield
            return
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            yield
        cur.wait_stream(self.stream)

    def forward_backward(self, app, mot, question, question_len, answers):
        """Forward, losses, backward of this rank's shard: leaves the (unreduced) gradient in gflat and the step's statistics
        in last_stats. Returns (total loss (device scalar), n_correct [B] int32)."""
        with self._on_stream():
            return self._forward_backward((app, mot), question, question_len, answers)

    @staticmethod
    def _run_model(model, feats, question, question_len):
        """feats: (app, mot) dense batches, or (DeviceFeatureStore, rows) -> the model's 7-tuple."""
        src, x = feats
        if isinstance(src, DeviceFeatureStore):
            return model.forward_from_store(src, x, question, question_len)
        return model(src, x, question, question_len)

    @staticmethod
    def _batch_dims(feats):
        """(B, N, device) of the batch that feats describes (see _run_model)."""
        src, x = feats
        if isinstance(src, DeviceFeatureStore):
            return x.shape[0], src.app.shape[1], x.device
        return src.shape[0], src.shape[1], src.device

    @staticmethod
    def _store_flags(feats):
        """The store's sticky out-of-range word joins the step flags: a step that read a bad row finalises to NaN."""
        return [feats[0].err] if isinstance(feats[0], DeviceFeatureStore) else []

    def _forward_backward_fp32(self, feats, question, question_len, answers):
        """fp32 mode (DualVGR.set_precision("fp32")): module-by-module forward, the auxiliary terms as ordinary autograd nodes
        on the fp32 graph outputs, gradients accumulated by autograd into the bound views of gflat (no deferred launches)."""
        model = self.model
        model.train()
        self.gflat.zero_()
        ag.begin_step_flags()
        unit = model.visual_input_unit
        B, N, _ = self._batch_dims(feats)
        outputs = self._run_model(model, feats, question, question_len)
        self.last_logits = outputs[0].detach()
        ce, correct = ag.CrossEntropyFn.apply(outputs[0], answers, False)
        loss, parts = ce, []
        if unit.layers > 0 and (self.alpha != 0 or self.beta != 0):
            c_com, c_dep = self._loss_coefs(B, N, unit.layers)
            for i in range(unit.layers):
                tot, vals = ag.AuxLossFn.apply(outputs[3][i], outputs[4][i], outputs[5][i], outputs[6][i], c_com, c_dep, False)
                loss = loss + tot
                parts.append(vals)
        loss.backward()
        self.last_stats = ops.finalize_loss(ce.detach().reshape(1), torch.stack(parts) if parts else None,
                                            self._store_flags(feats))
        return self.last_stats[0], correct

    def _forward_backward(self, feats, question, question_len, answers):
        """feats: (app, mot) or (DeviceFeatureStore, rows), see _run_model."""
        if ag.ACT[0] == torch.float32:
            return self._forward_backward_fp32(feats, question, question_len, answers)
        model = self.model
        model.train()
        B, N, dev = self._batch_dims(feats)
        # the 122 MB gradient buffer is cleared on a side stream, under the forward pass (nothing writes it before backward)
        cur = torch.cuda.current_stream()
        zs = fs.side_stream(dev, "aux")
        zs.wait_stream(cur)
        with torch.cuda.stream(zs):
            self.gflat.zero_()
            ev_zero = torch.cuda.Event()
            ev_zero.record()
        ag.begin_step_flags()
        ops.begin_step_counters(dev)               # zeroed tile counters of this step's dynamically scheduled GEMMs
        unit = model.visual_input_unit
        if self._reserve_env is None:
            ops.RESERVE_SMS[0] = min(64, 4 * ((B + 31) // 32))
        parts = None
        if unit.layers > 0 and (self.alpha != 0 or self.beta != 0):
            c_com, c_dep = self._loss_coefs(B, N, unit.layers)
            parts = torch.empty((unit.layers, B, 3), dtype=torch.float32, device=dev)
            unit._aux = (c_com, c_dep, parts)
        try:
            outputs = self._run_model(model, feats, question, question_len)
        finally:
            unit._aux = None
        self.last_logits = outputs[0].detach()
        ce, correct = ag.CrossEntropyFn.apply(outputs[0], answers, True)
        cur.wait_event(ev_zero)
        ops.DEFER_WGRAD[0] = True          # weight / bias gradients of the nn.Linear layers: queued during backward ...
        try:
            ce.backward()                  # the auxiliary terms' gradients are injected inside the unit stack's backward
        except BaseException:
            ops.clear_deferred()           # never leave half a step's gradients queued for the next one
            raise
        finally:
            ops.DEFER_WGRAD[0] = False
        ops.end_step_counters(dev)
        fs.join_side_streams(dev)          # question-encoder backward / auxiliary losses ran on side streams
        ops.flush_wgrads()                 # ... and launched as ONE grouped tcgen05 GEMM + grouped column sums
        ag._STEP_FLAGS.extend(self._store_flags(feats))
        self.last_stats = ops.finalize_loss(ce.detach(), parts, ag.step_flags())
        return self.last_stats[0], correct

    def loss_terms(self):
        """(total, loss_com_sum, loss_dep_sum) of the last step as train.py:148-154 accumulates them (un-scaled sums over the
        layers; host floats: this synchronises)."""
        s = [float(x) for x in self.last_stats.tolist()]
        unit = self.model.visual_input_unit
        B, N = self._last_BN
        c_com, c_dep = self._loss_coefs(B, N, unit.layers)
        com = s[1] / (c_com * B * N * N) if c_com != 0 else 0.0
        dep = s[2] / c_dep if c_dep != 0 else 0.0
        return s[0], com, dep

    def train_step(self, app, mot, question, question_len, answers):
        """One optimizer step on this rank's shard. Returns the (device) total loss of the shard."""
        self._last_BN = (app.shape[0], app.shape[1])
        with self._on_stream():
            total, _ = self._forward_backward((app, mot), question, question_len, answers)
            self._optimizer_step()
        return total

    def train_step_from_store(self, dstore, rows, question, question_len, answers):
        """train_step() on the batch (dstore.app[rows], dstore.mot[rows]) of a device-resident feature store
        (loader.DeviceFeatureStore), gathered inside the input prologue kernels. rows [B] int32 on the device. A row
        outside [0, V) sets dstore.err, and while that word is set every step's loss is NaN."""
        self._last_BN = (rows.shape[0], dstore.app.shape[1])
        with self._on_stream():
            total, _ = self._forward_backward((dstore, rows), question, question_len, answers)
            self._optimizer_step()
        return total

    def optimizer_step(self):
        with self._on_stream():
            self._optimizer_step()

    def _optimizer_step(self):
        if self.world > 1 and not self.skip_allreduce:
            if self._overlap is not None and self._overlap.fired:
                # the early bucket is already in flight on the side stream (launched from the backward pass); reduce the
                # encoders' bucket here and join
                dist.all_reduce(self.gflat[:self.late_numel], op=dist.ReduceOp.SUM, group=self.pg)
                torch.cuda.current_stream().wait_stream(self._overlap.side)
                self._overlap.fired = False
            else:
                dist.all_reduce(self.gflat, op=dist.ReduceOp.SUM, group=self.pg)
        self.step_count += 1
        self.step_dev += 1
        scale = 1.0 / self.world
        nsq = ops.sumsq(self.gflat)
        ops.adam_step(self.flat, self.gflat, self.m, self.v, self.lr, self.step_count, self.betas[0], self.betas[1],
                      self.eps, max_norm=self.max_norm, norm_sq=nsq, grad_scale=scale, step_dev=self.step_dev,
                      shadow=self.shadow)
        ag.invalidate_weight_cache()

    def dependency_poll_timeouts(self):
        """Number of step flags that were set in the last step, max over ranks: LSTM dependency polls that gave up and, in a
        step fed from a DeviceFeatureStore, the store's out-of-range-row word (0 in a healthy run; a non-zero value also
        turned that step's loss into NaN). Synchronises."""
        t = torch.zeros(1, device=self.flat.device) if self.last_stats is None else self.last_stats[3:4].clone()
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.pg)
        return int(t.item())

    # ------------------------------------------------------------------------------------------------------------
    # whole-step CUDA graph: forward, losses, backward, all-reduce, clip + Adam, weight re-casts = ONE graph launch.
    # Everything that changes between steps lives on the device (inputs in static buffers, dropout seed offset, Adam step).
    # NOTE: capture() runs `warmup` REAL optimizer steps on the given batch before recording (kernel attribute setup, NCCL
    # channel setup and allocator warm-up must not happen during capture): the parameters move, as with any train step.
    def capture(self, app, mot, question, question_len, answers, warmup=3):
        """Records one whole train step (forward, losses, backward, all-reduce, clip + Adam) as a CUDA graph over static
        input buffers; afterwards: load_batch(...) + replay(). NOTE: the `warmup` eager steps that precede the capture are
        REAL optimizer steps on the given batch (they warm the allocator, the weight caches and the side streams); pass the
        first training batch, or warmup=0 after at least one eager train_step()."""
        def step(st):
            return self.train_step(st["app"], st["mot"], st["q"], st["qlen"], st["ans"])
        return self._capture(dict(app=app, mot=mot, q=question, qlen=question_len, ans=answers), step, warmup)

    def capture_from_store(self, dstore, rows, question, question_len, answers, warmup=3):
        """capture() for train_step_from_store: the graph's static inputs are the rows and the question / answer tensors
        only (no feature buffers); afterwards load_rows(...) + replay(). The `warmup` eager steps are real optimizer steps."""
        def step(st):
            return self.train_step_from_store(dstore, st["rows"], st["q"], st["qlen"], st["ans"])
        return self._capture(dict(rows=rows, q=question, qlen=question_len, ans=answers), step, warmup)

    def _capture(self, named, step, warmup):
        from . import _lib
        self.static = {k: torch.empty_like(v) for k, v in named.items()}
        for k, v in named.items():
            self.static[k].copy_(v)
        _lib.lib.dvgr_set_seed_offset(self.seed_dev.data_ptr())
        self._seed_owner = True

        def body():
            self.seed_dev += 1
            return step(self.static)

        side = self.stream
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.cuda.graph(self.graph, stream=side):
            self.static_loss = body()
        self.launches_per_replay = _lib.launch_count() - n0    # library kernels recorded into the graph
        self.step_count = int(self.step_dev.item())            # capture itself executed no step: resync with the device
        ag.invalidate_weight_cache()
        return self.graph

    def release_static(self):
        self.graph = None
        self.static = None
        self.static_loss = None

    def close(self):
        """Detaches the engine from the library / autograd layer (call before dropping the engine)."""
        from . import _lib
        if getattr(self, "_seed_owner", False):
            _lib.lib.dvgr_set_seed_offset(None)
            self._seed_owner = False
        self.graph = None
        for p in self.params:
            ag.SHADOW.pop(id(p), None)
        _LIVE_ENGINES.discard(self)
        if not len(_LIVE_ENGINES):
            ag.DIRECT_GRAD[0] = False

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_batch(self, app, mot, question, question_len, answers, non_blocking=True):
        st = self.static
        for k, v in dict(app=app, mot=mot, q=question, qlen=question_len, ans=answers).items():
            st[k].copy_(v, non_blocking=non_blocking)

    def load_rows(self, rows, question, question_len, answers, non_blocking=True):
        """The next batch of a capture_from_store() graph: B video rows (int32) and the question / answer tensors."""
        st = self.static
        for k, v in dict(rows=rows, q=question, qlen=question_len, ans=answers).items():
            st[k].copy_(v, non_blocking=non_blocking)

    def replay(self):
        """One captured train step on the batch currently in the static buffers; returns the (device) loss tensor."""
        self.graph.replay()
        self.step_count += 1
        return self.static_loss

    # ------------------------------------------------------------------------------------------------------------
    def dp_parity_check(self, orc, cfg, samples_per_rank=16):
        """Data-parallel correctness on hardware (SURVEY §8e): every rank runs forward/backward on ITS shard of a seeded
        global batch, the flat gradients are all-reduced and averaged; every rank also runs the WHOLE batch alone with the
        single-process loss scaling; the two flat gradients must agree. Dropout off; the classifier's BatchNorm uses global
        batch statistics in the sharded run (sync_bn, forced on for this check) so the two computations are the same function.
        Also compares a parameter checksum across ranks. Returns a dict (rel-L2, checksum spread)."""
        model, dev = self.model, self.flat.device
        W, r = self.world, self.rank
        Bg = samples_per_rank * W
        app, mot, q, qlen, ans = orc.make_inputs(Bg, cfg["N"], cfg["L"], cfg["A"], cfg["V"], seed=77)
        saved = []
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):
                saved.append((m, "p", m.p)); m.p = 0.0
            if hasattr(m, "dropout") and isinstance(getattr(m, "dropout"), float):
                saved.append((m, "dropout", m.dropout)); m.dropout = 0.0
        ou = model.output_unit
        bn = ou.classifier[3]
        bn_state = (bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone())
        old = (self.world, ou.sync_bn_group, ou.sync_bn_world, self._overlap, model._unit_inputs_grad_hook if hasattr(model, "_unit_inputs_grad_hook") else None)
        try:
            model._unit_inputs_grad_hook = None
            self._overlap = None
            grp = self.pg if self.pg is not None else dist.group.WORLD
            sl = slice(r * samples_per_rank, (r + 1) * samples_per_rank)
            shard = [t[sl].to(dev) for t in (app, mot, q, qlen, ans)]
            full = [t.to(dev) for t in (app, mot, q, qlen, ans)]
            self._last_BN = (samples_per_rank, cfg["N"])
            rels = {}
            ab = (self.alpha, self.beta)
            for name, (al, be) in (("ce", (0.0, 0.0)), ("full", ab)):
                self.alpha, self.beta = al, be
                self.world, ou.sync_bn_group, ou.sync_bn_world = W, grp, W
                self.forward_backward(*shard)
                dist.all_reduce(self.gflat, op=dist.ReduceOp.SUM, group=self.pg)
                g_dp = (self.gflat / W).clone()
                # single-process reference on the concatenated batch
                ou.sync_bn_group, ou.sync_bn_world = None, 1
                self.world = 1
                self.forward_backward(*full)
                rels[name] = float((g_dp - self.gflat).norm() / self.gflat.norm().clamp_min(1e-30))
            self.alpha, self.beta = ab
        finally:
            self.world, ou.sync_bn_group, ou.sync_bn_world, self._overlap, hook = old
            model._unit_inputs_grad_hook = hook
            for m, name, val in saved:
                setattr(m, name, val)
            with torch.no_grad():
                bn.running_mean.copy_(bn_state[0]); bn.running_var.copy_(bn_state[1]); bn.num_batches_tracked.copy_(bn_state[2])
        chk = self.flat.double().sum().reshape(1)
        gathered = [torch.zeros_like(chk) for _ in range(W)]
        dist.all_gather(gathered, chk, group=self.pg)
        vals = [float(t) for t in gathered]
        return {"grad_rel_l2": rels["ce"], "grad_rel_l2_full_loss": rels["full"], "global_batch": Bg,
                "param_checksum_spread": max(vals) - min(vals),
                "note": "all-reduced, averaged flat gradient of the sharded step vs ONE rank on the concatenated batch; dropout off, "
                        "classifier BatchNorm on global statistics (sync) in the sharded run; grad_rel_l2 = cross-entropy loss "
                        "(deterministic up to bf16 / atomic order), grad_rel_l2_full_loss adds the ill-conditioned auxiliary terms "
                        "(their gradient differs by ~1e-3..1e-2 between two runs of the SAME computation, SURVEY 7)"}
