"""Generates tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference, CPU) on seeded
synthetic inputs and the deterministic weights of oracle/dualvgr_oracle.make_state_dict.  Runs only in the build
container; the fixtures it writes are what pins the oracle (and, through it, the CUDA path) to the reference.

    python oracle/make_golden.py [name ...]  # rewrites every fixture (or only the named ones)

Stored per config: the reference's outputs in float64 ("truth") and float32 (to record the reference's own
fp32-vs-fp64 floor), loss terms, and per-parameter gradient summaries (L2 norm + projection on a seeded probe vector)
for the CE-only loss and for the full training loss of train.py:146-154. A config with embed_samples keeps the aq/mq
embeddings of that many seeded batch rows only ("embed_rows" holds their indices)."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import dualvgr_oracle as orc   # noqa: E402
import ref_shim                # noqa: E402

CONFIGS = {
    # name: B, N, L, A, V, U, full tensors stored?
    "g1_B4_N8_U2": dict(B=4, N=8, L=7, A=10, V=30, U=2, full=True),
    "g2_B3_N20_U3": dict(B=3, N=20, L=9, A=32, V=50, U=3, full=False),
    "g3_B5_N16_U1": dict(B=5, N=16, L=5, A=17, V=40, U=1, full=False),
    # a realistic batch for the train-mode BatchNorm (the three above have 3-5 samples): holds the un-relaxed 2e-2 gradient gate
    "g4_B16_N20_U3": dict(B=16, N=20, L=12, A=32, V=60, U=3, full=False, embed_samples=6),
}


def embed_rows(B, k):
    """The batch rows whose aq/mq embeddings a fixture keeps when its config sets embed_samples (keeps the file < 1 MB)."""
    return np.sort(np.random.default_rng(0).choice(B, k, replace=False))


def no_dropout(model):
    for m in model.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
        if hasattr(m, "dropout") and isinstance(getattr(m, "dropout"), float):
            m.dropout = 0.0


def probe(name, shape, seed=4242):
    g = torch.Generator().manual_seed(seed + (hash_name(name) % 100000))
    return torch.randn(shape, generator=g, dtype=torch.float64)


def hash_name(name):
    h = 0
    for ch in name:
        h = (h * 131 + ord(ch)) % 1000003
    return h


def run_reference(modelset, losses, cfg, dtype, training):
    sd = orc.make_state_dict(cfg["U"], cfg["A"], cfg["V"])
    vocab = orc.make_vocab(cfg["V"], cfg["A"])
    model = modelset.DualVGR(vocab=vocab, num_of_nodes=cfg["N"], graph_module="GAT", graph_layers=1,
                             unit_layers=cfg["U"])
    model.load_state_dict(sd, strict=True)
    no_dropout(model)
    model = model.to(dtype)
    model.train(training)
    app, mot, q, qlen, ans = orc.make_inputs(cfg["B"], cfg["N"], cfg["L"], cfg["A"], cfg["V"])
    out = model(app.to(dtype), mot.to(dtype), q, qlen)
    return model, out, ans


def grads_summary(model):
    res = {}
    for name, p in model.named_parameters():
        g = p.grad.detach().double() if p.grad is not None else torch.zeros_like(p, dtype=torch.float64)
        res[name] = (float(g.norm()), float((g * probe(name, g.shape)).sum()))
    return res


def main():
    modelset = ref_shim.load_reference("cpu")
    losses = ref_shim.load_reference_losses()
    torch.Tensor.cuda = lambda self, *a, **k: self      # utils.py:22 hard-codes .cuda(); CPU run
    out_dir = os.path.join(os.path.dirname(HERE), "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    only = set(sys.argv[1:])
    for name, cfg in CONFIGS.items():
        if only and name not in only:
            continue
        blob = {"cfg": np.array([cfg[k] for k in ("B", "N", "L", "A", "V", "U")], dtype=np.int64)}
        # "bf16" = the reference's OWN reduced-precision execution: fp32 modules under torch.autocast(bfloat16) — the floor a
        # bf16 implementation of the path is judged against where the float64 truth is out of reach for ANY bf16 arithmetic
        # (the auxiliary losses centre nearly identical node embeddings, SURVEY.md §7)
        for dt_name, dtype in (("f64", torch.float64), ("f32", torch.float32), ("bf16", torch.float32)):
            torch.set_default_dtype(dtype)     # utils.py:22 builds R with the default dtype (torch.eye)
            amp = torch.autocast("cpu", dtype=torch.bfloat16, enabled=(dt_name == "bf16"))
            # ---- eval mode forward
            with amp:
                model, out, ans = run_reference(modelset, losses, cfg, dtype, training=False)
            blob[f"{dt_name}_logits_eval"] = out[0].detach().double().numpy()
            # ---- train mode forward + losses + grads
            with amp:
                model, out, ans = run_reference(modelset, losses, cfg, dtype, training=True)
                logits, aq_embed, mq_embed, ca, cm, aq, mq = out
                if dt_name == "bf16":
                    logits = logits.float()
                ce = torch.nn.functional.cross_entropy(logits, ans)
                N = cfg["N"]
                dep = sum(losses.loss_dependence(aq[i], ca[i], N) + losses.loss_dependence(mq[i], cm[i], N)
                          for i in range(len(aq)))
                com = sum(losses.common_loss(ca[i], cm[i]) for i in range(len(aq)))
                total = ce + 1.0 * com / len(aq) + 1e-8 * dep / len(aq)
            blob[f"{dt_name}_logits_train"] = logits.detach().double().numpy()
            blob[f"{dt_name}_losses"] = np.array([float(total), float(ce), float(com), float(dep)])
            model.zero_grad()
            ce.backward(retain_graph=True)
            gs = grads_summary(model)
            blob[f"{dt_name}_grad_ce"] = np.array([gs[k] for k in sorted(gs)])
            model.zero_grad()
            total.backward()
            gs = grads_summary(model)
            blob[f"{dt_name}_grad_full"] = np.array([gs[k] for k in sorted(gs)])
            if dt_name == "f64":
                blob["grad_names"] = np.array(sorted(gs))
                keep = {"aq_embed": aq_embed, "mq_embed": mq_embed}
                if cfg.get("embed_samples"):
                    rows = embed_rows(cfg["B"], cfg["embed_samples"])
                    blob["embed_rows"] = rows
                    keep = {k: v[torch.from_numpy(rows)] for k, v in keep.items()}
                if cfg["full"]:
                    for i in range(len(aq)):
                        keep.update({f"com_app_{i}": ca[i], f"com_mot_{i}": cm[i], f"aq_fusion_{i}": aq[i],
                                     f"mq_fusion_{i}": mq[i]})
                for k, v in keep.items():
                    blob[f"f64_{k}"] = v.detach().float().numpy()
                # state_dict contract (key order, shapes) of the reference
                sdr = model.state_dict()
                blob["sd_keys"] = np.array(list(sdr.keys()))
                blob["sd_shapes"] = np.array([",".join(map(str, v.shape)) for v in sdr.values()])
        torch.set_default_dtype(torch.float32)
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **blob)
        f64, f32 = blob["f64_logits_train"], blob["f32_logits_train"]
        print(name, "written", os.path.getsize(path) // 1024, "KiB; ref fp32-vs-fp64 logits rel-L2 =",
              np.linalg.norm(f64 - f32) / np.linalg.norm(f64), "losses", blob["f64_losses"], blob["f32_losses"])


if __name__ == "__main__":
    main()
