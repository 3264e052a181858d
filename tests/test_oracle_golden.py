"""Pins the CPU oracle (oracle/dualvgr_oracle.py) to the reference: the fixtures under tests/golden/ were produced by
the UNMODIFIED reference modules (oracle/make_golden.py). Tolerances are relative to the reference's own float64 run;
the reference's float32-vs-float64 gap stored in the fixture is the noise floor."""
import numpy as np
import pytest
import torch

import dualvgr_oracle as orc

CONFIGS = ["g1_B4_N8_U2", "g2_B3_N20_U3", "g3_B5_N16_U1", "g4_B16_N20_U3"]


def _probe(name, shape, seed=4242):
    h = 0
    for ch in name:
        h = (h * 131 + ord(ch)) % 1000003
    g = torch.Generator().manual_seed(seed + (h % 100000))
    return torch.randn(shape, generator=g, dtype=torch.float64)


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _run_oracle(g, training, dtype=torch.float64):
    B, N, L, A, V, U = [int(x) for x in g["cfg"]]
    sd = orc.cast_state_dict(orc.make_state_dict(U, A, V), dtype)
    for v in sd.values():
        if v.is_floating_point():
            v.requires_grad_(True)
    app, mot, q, qlen, ans = orc.make_inputs(B, N, L, A, V)
    out = orc.dualvgr_forward(sd, U, app.to(dtype), mot.to(dtype), q, qlen, training=training)
    return sd, out, ans, N


@pytest.mark.parametrize("name", CONFIGS)
def test_state_dict_contract(golden, name):
    g = golden(name)
    B, N, L, A, V, U = [int(x) for x in g["cfg"]]
    sd = orc.make_state_dict(U, A, V)
    assert list(sd.keys()) != []
    ref_keys = [str(k) for k in g["sd_keys"]]
    ref_shapes = {k: s for k, s in zip(ref_keys, [str(s) for s in g["sd_shapes"]])}
    assert set(sd.keys()) == set(ref_keys)
    for k, v in sd.items():
        assert ",".join(map(str, v.shape)) == ref_shapes[k], k


@pytest.mark.parametrize("name", CONFIGS)
def test_forward_eval_matches_reference(golden, name):
    g = golden(name)
    _, out, _, _ = _run_oracle(g, training=False)
    assert _rel(out[0].detach().numpy(), g["f64_logits_eval"]) < 1e-9


@pytest.mark.parametrize("name", CONFIGS)
def test_forward_train_losses_and_grads_match_reference(golden, name):
    g = golden(name)
    sd, out, ans, N = _run_oracle(g, training=True)
    logits = out[0]
    assert _rel(logits.detach().numpy(), g["f64_logits_train"]) < 1e-9
    assert np.array_equal(logits.detach().numpy().argmax(1), g["f64_logits_train"].argmax(1))
    rows = g["embed_rows"] if "embed_rows" in g.files else slice(None)     # g4 keeps a seeded subset of the batch
    assert _rel(out[1].detach().numpy()[rows], g["f64_aq_embed"]) < 1e-6      # fixture stores float32
    assert _rel(out[2].detach().numpy()[rows], g["f64_mq_embed"]) < 1e-6
    if "f64_com_app_0" in g.files:
        for i in range(len(out[3])):
            for key, lst in (("com_app", out[3]), ("com_mot", out[4]), ("aq_fusion", out[5]), ("mq_fusion", out[6])):
                assert _rel(lst[i].detach().numpy(), g[f"f64_{key}_{i}"]) < 1e-6, (key, i)
    total, ce, com, dep = orc.train_loss(out, ans, N)
    ref_total, ref_ce, ref_com, ref_dep = g["f64_losses"]
    assert abs(float(ce) - ref_ce) < 1e-9 * abs(ref_ce)
    # the auxiliary losses are ill-conditioned (SURVEY.md §7): in float64 the restatement still agrees tightly
    assert abs(float(com) - ref_com) < 1e-6 * abs(ref_com)
    assert abs(float(dep) - ref_dep) < 1e-6 * abs(ref_dep)
    assert abs(float(total) - ref_total) < 1e-7 * abs(ref_total)

    names = [str(n) for n in g["grad_names"]]
    params = [sd[n] for n in names]
    for loss, key in ((ce, "f64_grad_ce"), (total, "f64_grad_full")):
        grads = torch.autograd.grad(loss, params, retain_graph=True, allow_unused=True)
        ref = g[key]
        got_norm = np.array([0.0 if gr is None else float(gr.norm()) for gr in grads])
        got_proj = np.array([0.0 if gr is None else float((gr * _probe(n, gr.shape)).sum()) for n, gr in zip(names, grads)])
        # global (concatenated) relative error + per-tensor with an absolute floor (mathematically-zero grads)
        assert _rel(got_norm, ref[:, 0]) < 1e-6, key
        assert _rel(got_proj, ref[:, 1]) < 1e-6, key
        floor = 1e-9 * np.abs(ref[:, 0]).max()
        assert np.all(np.abs(got_norm - ref[:, 0]) <= 1e-5 * np.abs(ref[:, 0]) + floor), key


def test_adjacency_matches_reference_probe():
    # SURVEY.md §0 [probe]: diag 2/(N+1), off-diag 1/(N+1)
    a = orc.build_adjacency(20)
    assert torch.allclose(a.diagonal(), torch.full((20,), 2 / 21.0))
    assert torch.allclose(a[0, 1:], torch.full((19,), 1 / 21.0))


def test_fully_masked_row_is_uniform():
    # SURVEY.md §0: a fully masked adjacency row yields uniform attention, not NaN
    sd = orc.make_state_dict(1, 4, 8)
    x = torch.randn(2, 5, 768)
    adj = torch.ones(5, 5)
    adj[2] = 0
    gate = torch.rand(2, 5)
    out = orc.punish_gat(sd, "acGCN", 0, x, adj, gate)
    assert torch.isfinite(out).all()
