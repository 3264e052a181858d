#!/usr/bin/env python
"""bench.py — DualVGR train-step throughput on N B200s of one node (contract: see the task statement / DESIGN.md §6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--dtype bf16|fp32]     our arm (sm_100a kernels)
  python bench.py --impl reference [...]                     the reference's CPU algorithm (oracle port) on host cores
  python bench.py --dump-outputs DIR [...]                   also write what the last timed step computed to DIR/*.npy

Default workload = BASELINE.json configs[1]: SVQA shapes, N=20 clips x 16 frames x 2048-d appearance + 2048-d motion, GloVe-300
question of L=20 tokens, unit_layers=3, batch 256 per GPU, bf16 activations, full train step (forward, CE + common + HSIC
losses, backward, gradient all-reduce, clip 12, Adam). --config selects the other BASELINE.json configs (msrvtt, msvd_u1..u5,
clip64); --scaling strong splits the config's batch over the ranks instead of giving every rank a full one.
Synthetic data, seeded weights.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the bench writes nothing into it

F_, DV = 16, 2048
CONFIGS = {
    "svqa": dict(name="SVQA config (svqa_DualVGR_20.yml shapes)", B=256, N=20, L=20, A=32, V=200, U=3),
    "msrvtt": dict(name="MSRVTT-QA config (msrvtt_qa_DualVGR_16.yml shapes, open-ended answer vocab)", B=256, N=16, L=20,
                   A=4002, V=8000, U=3),
    "clip64": dict(name="synthetic 64-clip videos", B=512, N=64, L=20, A=32, V=200, U=3),
}
for _u in range(1, 6):
    CONFIGS[f"msvd_u{_u}"] = dict(name="MSVD-QA config (msvd_qa_DualVGR.yml shapes)", B=1024, N=8, L=20, A=1854, V=4000, U=_u)
METRIC, UNIT = "dualvgr_train_samples_per_sec", "samples/s"


def workload_name(c, n_gpus, per_gpu):
    return (f"{c['name']}: N={c['N']} clips x {F_} frames x {DV}-d, L={c['L']}, A={c['A']}, unit_layers={c['U']}, "
            f"batch {per_gpu}/GPU x {n_gpus} GPU, full train step")


def step_flops(c, batch):
    """Algorithmic FLOPs of one train step (SURVEY.md §8d / BASELINE.md §4): backward = 2x forward, minus the input
    gradients of the two 2048-d projections (their inputs need none)."""
    N, L, U, A = c["N"], c["L"], c["U"], c["A"]
    fwd = N * (201.3 + 37.7) + N * 3.15 + L * 8.4 + U * (N * 9.44 + L * 1.18 + 1.0) + N * 1.97 + N * 1.18 + 3.5 + 0.0015 * A
    return (3.0 * fwd - N * (201.3 + 3.15)) * 1e6 * batch


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clock / throttle sampling DURING the timed region (recipe line of B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------- reference arm
def cpu_sample_size(c):
    """Both CPU legs (cpu_baseline of our arm, --impl reference) time the SAME bounded sample: the first min(B, 256) samples
    of the workload batch (the whole batch at the default config), ~5 s of host work per step."""
    return min(c["B"], 256)


def cpu_reference_step_rate(c, sample_B, steps, warmup, threads):
    """The reference's algorithm for the path (oracle port, fp32) on the host cores: full train step on a bounded sample."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dualvgr_oracle as orc
    torch.set_num_threads(threads)
    sd = orc.make_state_dict(c["U"], c["A"], c["V"])
    params = []
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k:
            v.requires_grad_(True)
            params.append(v)
    opt = torch.optim.Adam(params, lr=1e-4)
    app, mot, q, qlen, ans = orc.make_inputs(sample_B, c["N"], c["L"], c["A"], c["V"])
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        out = orc.dualvgr_forward(sd, c["U"], app, mot, q, qlen, training=True)
        total, ce, com, dep = orc.train_loss(out, ans, c["N"])
        total.backward()
        torch.nn.utils.clip_grad_norm_(params, 12)
        opt.step()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return sample_B / statistics.median(times), statistics.median(times)


def cpu_sample_note(c, sample_B, steps, warmup):
    return (f"oracle port (oracle/dualvgr_oracle.py, fp32, torch CPU) full train step on {sample_B} of the {c['B']} samples of "
            f"the workload batch, median of {steps} steps after {warmup} warm-up; the Python reference cannot travel to the GPU box")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    sample_B = cpu_sample_size(c)
    steps, warmup = max(1, args.steps), max(0, min(args.warmup, 1))
    rate, sec = cpu_reference_step_rate(c, sample_B, steps, warmup, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(c, args.gpus, c["B"]),
                   "note": "CPU arm: each step is a bounded sample of the workload (see cpu_baseline.sample)"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": cpu_sample_note(c, sample_B, steps, warmup)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------- our arm
def classify_kernels(prof):
    """Kernel launches of one profiled step by owner: ours (libdualvgr_b200.so), NCCL, ATen / other libraries."""
    counts = {"total": 0, "library": 0, "nccl": 0, "aten_or_other": 0, "memcpy_memset": 0}
    other = {}
    for ev in prof.events():
        if str(getattr(ev, "device_type", "")).endswith("CUDA") is False:
            continue
        name = ev.name
        low = name.lower()
        if low.startswith("memcpy") or low.startswith("memset"):
            counts["memcpy_memset"] += 1
            continue
        counts["total"] += 1
        if "dvgr" in name or name.startswith(("scatter_kernel", "colsum_grouped_kernel")):
            counts["library"] += 1
        elif "nccl" in low:
            counts["nccl"] += 1
        else:
            counts["aten_or_other"] += 1
            other[name[:60]] = other.get(name[:60], 0) + 1
    counts["aten_top"] = sorted(other.items(), key=lambda kv: -kv[1])[:6]
    return counts


DUMP_MAX_ELEMS = 1 << 22       # per array: 16 MB in float32, so the four arrays of --dump-outputs stay under 64 MB


def dump_outputs(out_dir, model, loss, logits):
    """--dump-outputs: what the last timed step handed its caller, as float32 DIR/<name>.npy: the loss, the logits, and
    the updated parameters and their gradients (every trainable parameter flattened, in the model's parameter order, so
    the files do not depend on the engine's buffer layout). An array above DUMP_MAX_ELEMS elements is replaced by its
    flattened elements at a fixed seeded sample of positions (the same positions for arrays of the same size)."""
    import numpy as np
    import torch

    def sample(t):
        t = t.detach()
        if t.numel() <= DUMP_MAX_ELEMS:
            return t
        idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
        return t.reshape(-1)[torch.from_numpy(idx).to(t.device)]

    params = [p for p in model.parameters() if p.requires_grad]
    arrays = {"loss": loss.reshape(1), "logits": logits,
              "params": torch.cat([p.detach().reshape(-1) for p in params]),
              "grads": torch.cat([p.grad.reshape(-1) for p in params])}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), sample(t).float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dualvgr_oracle as orc                      # ONLY make_state_dict / make_inputs / baselines (checker side)
    import dualvgr_videoqa_b200._lib as L
    import dualvgr_videoqa_b200.model.models as M
    from dualvgr_videoqa_b200.engine import TrainEngine
    from dualvgr_videoqa_b200 import autograd as ag

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to STDOUT when the first communicator is created; rank 0 must print exactly one
        # JSON line there, so file descriptor 1 points at stderr until the engine (and its first collective) exists
        sys.stdout.flush()
        saved_stdout_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    c = dict(CONFIGS[args.config])
    if args.batch:
        c["B"] = args.batch
    strong = args.scaling == "strong"
    Bl = c["B"] // world if strong else c["B"]          # samples on this rank
    torch.manual_seed(666)
    model = M.DualVGR(vocab=orc.make_vocab(c["V"], c["A"]), num_of_nodes=c["N"], graph_module="GAT", graph_layers=1,
                      unit_layers=c["U"])
    model.load_state_dict(orc.make_state_dict(c["U"], c["A"], c["V"]), strict=True)
    model = model.to(dev).train()
    if args.dtype == "fp32":
        model.set_precision("fp32")
    eng = TrainEngine(model, lr=1e-4, max_norm=12.0, alpha=1.0, beta=1e-8)
    if world > 1:
        torch.cuda.synchronize()
        sys.stdout.flush()
        os.dup2(saved_stdout_fd, 1)
        os.close(saved_stdout_fd)

    # synthetic shard of this rank, generated on the host, pinned; a device-resident copy for the kernel-side number
    g = torch.Generator().manual_seed(1000 + rank)
    host = {
        "app": torch.randn((Bl, c["N"], F_, DV), generator=g).abs_().pin_memory(),
        "mot": torch.randn((Bl, c["N"], DV), generator=g).abs_().pin_memory(),
    }
    qlen = torch.randint(5, c["L"] + 1, (Bl,), generator=g); qlen[0] = c["L"]
    q = torch.randint(2, c["V"], (Bl, c["L"]), generator=g) * (torch.arange(c["L"])[None] < qlen[:, None])
    host["q"], host["qlen"] = q.long().pin_memory(), qlen.long().pin_memory()
    host["ans"] = torch.randint(0, c["A"], (Bl,), generator=g).pin_memory()
    res = {k: v.to(dev) for k, v in host.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())

    # the warm-up (and capture) steps are real optimizer steps whose reductions are not bit-reproducible: the timed steps
    # start again from this seeded state, so that every run hands them the same weights and optimizer state
    state = [eng.flat, eng.m, eng.v, eng.step_dev, eng.seed_dev] + list(model.buffers())
    initial = [t.clone() for t in state]

    use_graph = not args.no_graph
    if use_graph:
        eng.capture(res["app"], res["mot"], res["q"], res["qlen"], res["ans"], warmup=max(3, args.warmup))

    def step_resident():
        if use_graph:
            return eng.replay()
        return eng.train_step(res["app"], res["mot"], res["q"], res["qlen"], res["ans"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        """n calls of fn bracketed by barrier + synchronize on both sides, CUDA events, max over ranks -> ms total."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        out = None
        for _ in range(n):
            out = fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    for _ in range(max(3, args.warmup)):
        step_resident()
    barrier()
    with torch.no_grad():
        for t, t0 in zip(state, initial):
            t.copy_(t0)
    eng.sync_shadow()
    eng.step_count = 0
    del state, initial
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = L.launch_count()
    ms_max, loss = timed(step_resident, args.steps)
    launches = L.launch_count() - n0
    if use_graph:
        launches = eng.launches_per_replay * args.steps      # kernels of libdualvgr_b200.so inside each replayed graph
    clocks = sampler.stop() if rank == 0 else None
    value = Bl * world * args.steps / (ms_max / 1e3)
    final_loss = float(loss)
    timeouts = eng.dependency_poll_timeouts()           # max over ranks; a non-zero value also poisons the loss with NaN
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, loss, eng.last_logits)

    # ---- who launched what: one profiled replay, kernels classified by owner (ours / NCCL / ATen)
    kernels = None
    if use_graph and not args.no_kernel_census:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.replay()
            torch.cuda.synchronize()
        kernels = classify_kernels(prof)

    # ---- data-parallel parity (N > 1): averaged flat gradient of the sharded step vs ONE rank on the concatenated batch
    dp_parity = None
    if world > 1 and not args.no_dp_parity:
        dp_parity = eng.dp_parity_check(orc, c, samples_per_rank=16)

    # ---- the dominant kernel — lstm_seq_fwd_kernel: the appearance encoder's input projection (K = 2048) and its 16
    #      recurrent steps (K = 384) fused in ONE persistent tcgen05 launch — timed live with CUDA events on its launching
    #      stream at the workload's exact shape; operands (335 MB of features, 503 MB of gates out) exceed the 126 MB L2
    import dualvgr_videoqa_b200.ops as ops
    T_, S_, H_ = F_, Bl * c["N"], 384
    xa = (torch.randn((T_, S_, DV), device=dev) * 0.5).to(torch.bfloat16)
    wih = (torch.randn((8 * H_, DV), device=dev) * 0.02).to(torch.bfloat16)
    whh = (torch.randn((2, 4 * H_, H_), device=dev) * 0.05).to(torch.bfloat16)
    bih = torch.zeros(8 * H_, device=dev)
    r_ = None
    for _ in range(3):
        r_ = None                                   # one output set live at a time: the caching allocator reuses its blocks,
        r_ = ops.lstm_seq_fwd(xa, wih, whh, bih)     # so no cudaMalloc lands between the two events below
    gemm_ms = []
    for _ in range(10):
        r_ = None
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); r_ = ops.lstm_seq_fwd(xa, wih, whh, bih); b.record()
        torch.cuda.synchronize()
        gemm_ms.append(a.elapsed_time(b))
        timeouts += int(r_[5][-1])
    del xa, r_

    # ---- e2e: same step through the public API with HOST buffers; H2D of every step's inputs inside the timed region
    #      (double-buffered on a copy stream, as an input pipeline would), D2H read of the loss every step
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    loss_host = torch.zeros(args.steps + 8, dtype=torch.float32).pin_memory()

    def measure_e2e(host_t):
        bufs = [{k: torch.empty_like(v, device=dev) for k, v in host_t.items()} for _ in range(2)]

        def prefetch(i):
            b = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[b])
                for k, v in host_t.items():
                    bufs[b][k].copy_(v, non_blocking=True)
                ready[b].record(copy_stream)

        def run_e2e(n):
            cur = torch.cuda.current_stream()
            for b in range(2):
                consumed[b].record(cur)
            prefetch(0)
            for i in range(n):
                if i + 1 < n:
                    prefetch(i + 1)
                b = i % 2
                cur.wait_event(ready[b])
                if use_graph:   # device-to-device hand-over of the staged batch into the graph's static inputs, then ONE launch
                    eng.load_batch(bufs[b]["app"], bufs[b]["mot"], bufs[b]["q"], bufs[b]["qlen"], bufs[b]["ans"])
                    consumed[b].record(cur)
                    lo = eng.replay()
                else:
                    lo = eng.train_step(bufs[b]["app"], bufs[b]["mot"], bufs[b]["q"], bufs[b]["qlen"], bufs[b]["ans"])
                    consumed[b].record(cur)
                loss_host[i].copy_(lo, non_blocking=True)

        run_e2e(2)
        ms, _ = timed(lambda: run_e2e(args.steps), 1)
        del bufs
        return Bl * world * args.steps / (ms / 1e3)

    e2e_value = e2e_bf16 = None
    h2d_bf16 = None
    if not args.no_e2e:
        e2e_value = measure_e2e(host)          # the reference's data format: fp32 features (DataLoader.py:61-84)
        if use_graph and not args.no_bf16_e2e:
            # informational second leg (SURVEY §8f.3): the same step with the features STORED as bf16 on the host, i.e. half
            # the bytes on the PCIe link, which is what bounds the fp32 leg; needs its own captured graph (bf16 prologue)
            host16 = dict(host)
            host16["app"] = host["app"].to(torch.bfloat16).pin_memory()
            host16["mot"] = host["mot"].to(torch.bfloat16).pin_memory()
            h2d_bf16 = sum(v.numel() * v.element_size() for v in host16.values())
            eng.graph = None
            res16 = {k: v.to(dev) for k, v in host16.items()}
            eng.capture(res16["app"], res16["mot"], res16["q"], res16["qlen"], res16["ans"], warmup=1)
            e2e_bf16 = measure_e2e(host16)
            del res16

    # ---- exposed all-reduce: the same step captured WITHOUT the gradient exchange, timed the same way. LAST leg: without the
    #      exchange the replicas drift apart, nothing after this point may depend on them
    allreduce_exposed_ms = None
    if world > 1 and use_graph and not args.no_comm_ab:
        eng.graph = None
        eng.skip_allreduce = True
        eng.capture(res["app"], res["mot"], res["q"], res["qlen"], res["ans"], warmup=1)
        eng.replay()
        ms_nocomm, _ = timed(eng.replay, args.steps)
        allreduce_exposed_ms = (ms_max - ms_nocomm) / args.steps
        eng.skip_allreduce = False
        eng.graph = None

    if rank == 0:
        pk = peaks()
        # algorithmic FLOPs (SURVEY §8d): W_ih product of both directions + the recurrent products of steps 1..T-1 (h_0 = 0)
        flops = 2.0 * (Bl * c["N"]) * (8 * 384) * (F_ * DV + (F_ - 1) * 384)
        gemm_avg = statistics.mean(gemm_ms) if gemm_ms else float("nan")
        achieved = flops / (gemm_avg * 1e-3) / 1e12 if gemm_ms else None
        traffic = None
        prof_path = os.path.join(ROOT, "profiles", "dominant_kernel.json")
        if os.path.exists(prof_path) and args.config == "svqa" and not args.batch:
            pj = json.load(open(prof_path))
            if str(pj.get("kernel", "")).startswith("lstm_seq_fwd_kernel"):     # only a capture of THIS kernel counts
                traffic = pj.get("dram_bytes_per_launch")
        sflops = step_flops(c, Bl)
        ms_step = ms_max / args.steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "bf16" if args.dtype == "bf16" else "f32 (3x bf16 split tensor-core products, fp32 activations)",
            "data": "synthetic",
            "config": {"workload": workload_name(c, world, Bl), "name": args.config,
                       "parallelism": f"dp{world}" if world > 1 else "single",
                       "l2": f"no explicit flush: each step streams {h2d_bytes / 1e6:.0f} MB of fp32 features + GBs of "
                             "intermediates, far above the 126 MB L2",
                       "optimizer": "clip 12 + Adam lr 1e-4 (flat fused)", "dropout": "on (train mode, reference rates)",
                       "cuda_graph": bool(use_graph), "final_loss": final_loss},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "note": "host buffers in the reference's format (fp32 features): bound by the host link, not by the kernels"},
            "e2e_bf16_features": {"value": e2e_bf16, "unit": UNIT, "h2d_bytes_per_step": h2d_bf16, "d2h_bytes_per_step": 4,
                                  "note": "informational: same step with the clip features stored as bf16 on the host"},
            "gpu_launches": int(launches),
            "kernels_per_step": kernels,
            "aten_launches_per_step": kernels["aten_or_other"] if kernels else None,
            "step_roofline": {"flop_per_step_per_gpu": sflops, "ms_at_sustained_peak": sflops / (pk["tf"] * 1e12) * 1e3,
                              "frac": sflops / (pk["tf"] * 1e12) * 1e3 / ms_step, "peak_tflops": pk["tf"]},
            "roofline": {"kernel": "lstm_seq_fwd_kernel<BN=256> (appearance encoder forward: W_ih product + 16 recurrent steps, one persistent launch)",
                         "bound": "tensor", "achieved": achieved, "peak": pk["tf_burst"], "unit": "TFLOP/s",
                         "frac": (achieved / pk["tf_burst"]) if achieved else None,
                         "frac_of_sustained_peak": (achieved / pk["tf"]) if achieved else None, "traffic": traffic,
                         "peak_source": pk["src"] + ", burst bf16 figure (the kernel is timed alone); the sustained figure is "
                                        f"{pk['tf']} TFLOP/s",
                         "timing": "mean of 10 isolated launches at the workload shape, CUDA events on the launch stream",
                         "launch_ms": gemm_avg, "dependency_poll_timeouts": timeouts},
            "dependency_poll_timeouts": timeouts,
        }
        if allreduce_exposed_ms is not None:
            line["allreduce_exposed_ms"] = allreduce_exposed_ms
        if dp_parity is not None:
            line["dp_parity"] = dp_parity["grad_rel_l2"]
            line["dp_parity_detail"] = dp_parity
        if world == 1 and not args.no_eager:
            # the like-for-like GPU number (SURVEY §8d, BASELINE.md §5.2): PyTorch eager on this B200, same batch, full step
            eng.graph = None
            eng.release_static()
            torch.cuda.empty_cache()
            import eager_gpu
            eg = {"unit": UNIT, "note": "oracle/eager_gpu.py: the reference's eager execution restated on the oracle's formulas "
                                        "with cuDNN LSTMs; 'faithful' keeps the reference's pair tensor, .cpu() round trips and "
                                        "per-sample loops, 'lean' drops them (faster than the reference can be); dropout on, "
                                        "CUDA events, median of 3 steps after 2 warm-up"}
            batch = (res["app"], res["mot"], res["q"], res["qlen"], res["ans"])
            for key, kw in (("lean_fp32", dict()), ("lean_bf16_autocast", dict(autocast=True)), ("faithful_fp32", dict(faithful=True))):
                try:
                    ms_e, rate_e = eager_gpu.time_eager_step(c, batch, **kw)
                    eg[key] = {"value": rate_e, "ms_per_step": ms_e}
                except Exception as ex:      # e.g. out of memory at the 64-clip config (the [B,N,N,2Dh] pair tensor)
                    eg[key] = {"value": None, "error": f"{type(ex).__name__}: {str(ex)[:120]}"}
                    torch.cuda.empty_cache()
            line["eager_gpu_baseline"] = eg
        if world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            sB = cpu_sample_size(c)
            rate, sec = cpu_reference_step_rate(c, sB, 2, 1, threads)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": cpu_sample_note(c, sB, 2, 1)}
        print(json.dumps(line), flush=True)
    if world > 1:
        # the captured graph holds NCCL work objects; tearing the communicator down under it can block forever, so
        # synchronise, drop the graph, and leave without the (optional) destroy_process_group handshake
        dist.barrier()
        torch.cuda.synchronize()
        eng.close()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    if os.environ.get("DVGR_HANG_DUMP"):          # debugging aid: dump all Python stacks if the run stalls
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["DVGR_HANG_DUMP"]), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="svqa", choices=sorted(CONFIGS), help="BASELINE.json workload (default: configs[1])")
    ap.add_argument("--batch", type=int, default=0, help="override the config's batch")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the config's batch on EVERY rank; strong: the config's batch split over the ranks")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"], help="fp32 = the 1e-4 parity mode (3x bf16 split products)")
    ap.add_argument("--no-e2e", action="store_true", help="profiling aid: skip the host-buffer e2e leg")
    ap.add_argument("--no-bf16-e2e", action="store_true", help="skip the informational e2e leg with bf16-stored features")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of replaying the captured CUDA graph")
    ap.add_argument("--no-cpu", action="store_true", help="profiling aid: skip the cpu_baseline leg")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager GPU baseline leg")
    ap.add_argument("--no-kernel-census", action="store_true", help="skip the profiled replay that counts kernels by owner")
    ap.add_argument("--no-comm-ab", action="store_true", help="N>1: skip the second capture that measures the exposed all-reduce")
    ap.add_argument("--no-dp-parity", action="store_true", help="N>1: skip the sharded-vs-single-rank gradient check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss, logits, parameters and "
                    "gradients to DIR/*.npy (float32; seeded samples of the large ones) to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA arm (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
