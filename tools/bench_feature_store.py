"""Train / validate from a device-resident feature store vs the host input pipeline, at the SVQA config on one GPU.

Legs (alternated, each repeated --reps times; one rep = one shuffled epoch of --batches-per-epoch captured train steps, with
a D2H copy of every step's loss):
  a_store_fp32  loader.DeviceBatchLoader on a DeviceFeatureStore of fp32 features (TrainEngine.capture_from_store)
  b_store_bf16  the same on a bf16 store
  c_host_pinned loader.PinnedBatchLoader from the host FeatureStore (fp32), TrainEngine.capture + load_batch
Validation: EvalEngine fed by (a) vs EvalEngine fed by PinnedBatchLoader, same rep structure. Also: the appearance prologue
alone (CUDA events; gathered from the store at shuffled rows vs dense over a resident batch), store size and upload time, and
the GPU's name and power limit read in the same run. The synthetic store has --videos videos (default 1024, 2.7 GB fp32:
far above the 126 MB L2). Prints one JSON line (and writes it to --out when given).

    python tools/bench_feature_store.py [--videos 1024] [--reps 3] [--batches-per-epoch 12] [--out FILE]"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_max_mhz": float(out[1])}
    except Exception as e:      # the numbers are reported as missing, never guessed
        return {"name": name, "power_limit_w": None, "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--batches-per-epoch", type=int, default=12)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prologue-launches", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_feature_store: needs a CUDA device")
    import dualvgr_oracle as orc
    import dualvgr_videoqa_b200.model.models as M
    import dualvgr_videoqa_b200.ops as ops
    from dualvgr_videoqa_b200.engine import TrainEngine
    from dualvgr_videoqa_b200.evaluate import EvalEngine, SVQA_CATEGORIES
    from dualvgr_videoqa_b200.loader import DeviceBatchLoader, DeviceFeatureStore, FeatureStore, PinnedBatchLoader

    torch.manual_seed(0)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    B, N, F, Dv, L, A, Vq, U = args.batch, 20, 16, 2048, 20, 32, 200, 3          # BASELINE configs[1] (SVQA)
    V = args.videos
    g = np.random.default_rng(0)
    app = g.random((V, N, F, Dv), dtype=np.float32)
    mot = g.random((V, N, Dv), dtype=np.float32)
    host32 = FeatureStore(app, mot)
    app16 = np.empty(app.shape, dtype=np.uint16)
    for v0 in range(0, V, 64):                       # chunked: the conversion's temporaries stay small
        app16[v0:v0 + 64] = FeatureStore.to_bf16_bits(app[v0:v0 + 64])
    host16 = FeatureStore(app16, FeatureStore.to_bf16_bits(mot))
    S = B * args.batches_per_epoch
    qlen = g.integers(3, L + 1, S)
    samples = {"video_idx": g.integers(0, V, S), "question": g.integers(2, Vq, (S, L)) * (np.arange(L)[None] < qlen[:, None]),
               "question_len": qlen, "answer": g.integers(0, A, S)}
    samples_eval = dict(samples, category=g.integers(0, 15, S))

    res = {"config": {"batch": B, "N": N, "F": F, "Dv": Dv, "U": U, "videos": V, "steps_per_rep": args.batches_per_epoch,
                      "reps": args.reps}}
    stores = {}
    for name, host in (("fp32", host32), ("bf16", host16)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stores[name] = DeviceFeatureStore(host, dev)
        torch.cuda.synchronize()
        res[f"store_{name}"] = {"bytes": stores[name].nbytes, "upload_s": time.perf_counter() - t0}

    # ---- prologue alone: gathered at shuffled rows vs dense over a resident batch (CUDA events, many launches)
    rows_all = torch.from_numpy(g.integers(0, V, (args.prologue_launches, B)).astype(np.int32)).to(dev)
    dense = torch.from_numpy(app[:B]).to(dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)

    def ev_time(fn):
        fn(0)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(args.prologue_launches):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / args.prologue_launches

    pro = {}
    for rep in range(args.reps):
        for key, fn in (
                ("gather_fp32", lambda i: ops.prep_features_gather(stores["fp32"].app, rows_all[i], F, True, True, 0.15, 1, 0, err)),
                ("gather_bf16", lambda i: ops.prep_features_gather(stores["bf16"].app, rows_all[i], F, True, True, 0.15, 1, 0, err)),
                ("dense_fp32", lambda i: ops.prep_features(dense.view(-1, Dv), F, True, True, 0.15, 1, 0))):
            pro.setdefault(key, []).append(ev_time(fn))
    res["appearance_prologue_ms"] = pro
    res["appearance_prologue_bytes_read"] = {"fp32": B * N * F * Dv * 4, "bf16": B * N * F * Dv * 2}
    del dense

    # ---- train legs
    base = M.DualVGR(vocab=orc.make_vocab(Vq, A), num_of_nodes=N, graph_module="GAT", graph_layers=1, unit_layers=U)
    base.load_state_dict(orc.make_state_dict(U, A, Vq), strict=True)
    loss_host = torch.zeros(args.batches_per_epoch, dtype=torch.float32).pin_memory()
    legs = {}
    for key, store in (("a_store_fp32", stores["fp32"]), ("b_store_bf16", stores["bf16"])):
        eng = TrainEngine(copy.deepcopy(base).to(dev), lr=1e-4)
        loader = DeviceBatchLoader(store, samples, B, dev, shuffle=True, seed=1)
        legs[key] = (eng, lambda eng=eng, loader=loader, store=store: train_epoch_store(eng, loader, store, loss_host))
    eng_c = TrainEngine(copy.deepcopy(base).to(dev), lr=1e-4)
    loader_c = PinnedBatchLoader(host32, samples, B, dev, shuffle=True, seed=1)
    legs["c_host_pinned"] = (eng_c, lambda: train_epoch_pinned(eng_c, loader_c, loss_host))
    for _, run in legs.values():          # capture (3 warm-up steps) + one untimed epoch per leg
        run()
    rates, finite = {k: [] for k in legs}, {k: True for k in legs}
    for rep in range(args.reps):
        for key, (_, run) in legs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run()
            torch.cuda.synchronize()
            rates[key].append(S / (time.perf_counter() - t0))
            finite[key] &= bool(np.isfinite(loss_host.numpy()).all())
    res["train_samples_per_s"] = rates
    res["train_losses_finite"] = finite
    res["dependency_poll_timeouts"] = {k: e.dependency_poll_timeouts() for k, (e, _) in legs.items()}
    for e, _ in legs.values():
        e.close()
    del legs, eng_c

    # ---- validation: (a) vs EvalEngine fed by PinnedBatchLoader
    model = copy.deepcopy(base).to(dev).eval()
    ev_a, ev_c = EvalEngine(model, SVQA_CATEGORIES), EvalEngine(model, SVQA_CATEGORIES)
    ld_a = DeviceBatchLoader(stores["fp32"], samples_eval, B, dev)
    ld_c = PinnedBatchLoader(host32, samples_eval, B, dev)

    def eval_a():
        for rows, q, ql, ans, cat in ld_a:
            if ev_a.graph is None:
                ev_a.capture_from_store(stores["fp32"], rows, q, ql, ans, cat)
            ev_a.load_rows(rows, q, ql, ans, cat)
            ev_a.replay()

    def eval_c():
        for ap_, mo, q, ql, ans, cat in ld_c:
            if ev_c.graph is None:
                ev_c.capture(ap_, mo, q, ql, ans, cat)
            ev_c.load_batch(app=ap_, mot=mo, q=q, qlen=ql, ans=ans, cat=cat)
            ev_c.replay()

    evals = {"a_store_fp32": eval_a, "c_host_pinned": eval_c}
    for fn in evals.values():
        fn()
    ev_a.reset(); ev_c.reset()
    eval_rates = {k: [] for k in evals}
    for rep in range(args.reps):
        for key, fn in evals.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            eval_rates[key].append(S / (time.perf_counter() - t0))
    res["eval_samples_per_s"] = eval_rates
    res["eval_counts_equal"] = ev_a.result()["counts"] == ev_c.result()["counts"]
    res["store_error_words"] = {k: s.read_error() for k, s in stores.items()}
    res["gpu"] = gpu_identity()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


def train_epoch_store(eng, loader, store, loss_host):
    for i, (rows, q, ql, ans) in enumerate(loader):
        if eng.graph is None:
            eng.capture_from_store(store, rows, q, ql, ans, warmup=3)
        eng.load_rows(rows, q, ql, ans)
        loss_host[i].copy_(eng.replay(), non_blocking=True)


def train_epoch_pinned(eng, loader, loss_host):
    for i, (ap_, mo, q, ql, ans) in enumerate(loader):
        if eng.graph is None:
            eng.capture(ap_, mo, q, ql, ans, warmup=3)
        eng.load_batch(ap_, mo, q, ql, ans)
        loss_host[i].copy_(eng.replay(), non_blocking=True)


if __name__ == "__main__":
    main()
