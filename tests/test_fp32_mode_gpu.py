"""fp32 mode (north_star: "within 1e-4 relative error in fp32"): the 3 x bf16 split products on the tcgen05 GEMM, the fp32
variants of the fused kernels, the fp32 LSTM path, and the whole model against the float64 oracle at 1e-4."""
import pytest
import torch

import dualvgr_oracle as orc

pytestmark = pytest.mark.gpu
BF16, F32 = torch.bfloat16, torch.float32


def rel(a, b):
    import numpy as np
    a, b = (torch.as_tensor(np.asarray(t), dtype=torch.float64) if not torch.is_tensor(t) else t.detach().double().cpu()
            for t in (a, b))
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.fixture(scope="module")
def ops():
    import dualvgr_videoqa_b200.ops as ops
    import dualvgr_videoqa_b200._lib as L
    L.lib.dvgr_set_seed_offset(None)
    return ops


@pytest.mark.parametrize("M,N,K", [(300, 768, 768), (1000, 136, 300), (257, 3072, 2048)])
def test_split_products_reach_fp32_accuracy(ops, M, N, K):
    """x W^T, dy W and dy^T x from bf16 planes [lo | hi | hi]: a_lo b_hi + a_hi b_hi + a_hi b_lo in ONE launch each,
    against float64; a single bf16 pass sits at ~3e-3."""
    g = torch.Generator().manual_seed(M + N + K)
    x = torch.randn((M, K), generator=g).cuda()
    w = (torch.randn((N, K), generator=g) * 0.05).cuda()
    b = torch.randn(N, generator=g).cuda()
    dy = torch.randn((M, N), generator=g).cuda()
    x3, w3, dy3 = ops.split3(x), ops.split3(w), ops.split3(dy)
    assert rel(x3[0].float()[:, :K] + x3[1].float()[:, :K], x) < 2e-5 and torch.equal(x3[1], x3[2])
    y = torch.empty((M, N), dtype=F32, device="cuda")
    ops.gemm3(x3, 0, w3, 0, M, N, K, y, bias=b, act="elu")
    ref = torch.nn.functional.elu(x.double() @ w.double().t() + b.double())
    assert rel(y, ref) < 2e-5, rel(y, ref)
    y1 = ops.linear_fwd(x.to(BF16) if K % 8 == 0 else torch.nn.functional.pad(x, (0, (-K) % 8)).to(BF16),
                        w.to(BF16) if K % 8 == 0 else torch.nn.functional.pad(w, (0, (-K) % 8)).to(BF16), bias=b, act="elu",
                        out_dtype=F32)
    assert rel(y1, ref) > 20 * rel(y, ref)                                    # the split really buys two orders of magnitude
    dx = torch.empty((M, K), dtype=F32, device="cuda")
    ops.gemm3(dy3, 0, w3, 1, M, K, N, dx)                                     # dgrad: W read MN-major
    assert rel(dx, dy.double() @ w.double()) < 2e-5
    dw = torch.zeros((N, K), dtype=F32, device="cuda")
    ops.gemm3(dy3, 1, x3, 1, N, K, M, dw)                                     # wgrad: both MN-major
    assert rel(dw, dy.double().t() @ x.double()) < 2e-5
    ops.gemm3(dy3, 1, x3, 1, N, K, M, dw, beta=True)                          # accumulate
    assert rel(dw, 2 * (dy.double().t() @ x.double())) < 2e-5


# ------------------------------------------------------------------------------------------------- fp32 recurrent path
@pytest.mark.parametrize("T,S,K,H,ragged", [(5, 37, 48, 32, False), (9, 21, 300, 64, True)])
def test_lstm32_matches_torch_float64(ops, T, S, K, H, ragged):
    """fp32_path.Lstm32Fn (split products + fp32 cells, 4 directions = two BiLSTMs over one input) against nn.LSTM in
    float64 on the CPU, packed-sequence semantics for ragged lengths: outputs and every gradient at 1e-4."""
    import dualvgr_videoqa_b200.fp32_path as f32
    g = torch.Generator().manual_seed(T * 100 + S)
    x = torch.randn((S, T, K), generator=g) * 0.7
    lens = torch.randint(1, T + 1, (S,), generator=g) if ragged else torch.full((S,), T)
    if ragged:
        lens[0] = T
    refs = [torch.nn.LSTM(K, H, batch_first=True, bidirectional=True).double() for _ in range(2)]
    for m in refs:
        for p in m.parameters():
            torch.nn.init.uniform_(p, -0.3, 0.3, generator=g)
    xr = x.double().requires_grad_(True)
    seqs, lasts = [], []
    for m in refs:
        pk = torch.nn.utils.rnn.pack_padded_sequence(xr, lens, batch_first=True, enforce_sorted=False)
        o, (hn, _) = m(pk)
        o, _ = torch.nn.utils.rnn.pad_packed_sequence(o, batch_first=True, total_length=T)
        seqs.append(o); lasts.append(torch.cat([hn[0], hn[1]], -1))
    ref_seq, ref_last = torch.cat(seqs, -1), torch.cat(lasts, -1)
    w_seq, w_last = torch.randn(ref_seq.shape, generator=g).double(), torch.randn(ref_last.shape, generator=g).double()
    ((ref_seq * w_seq).sum() + (ref_last * w_last).sum()).backward()

    params = []
    for m in refs:
        for sfx in ("", "_reverse"):
            params += [getattr(m, f"{n}_l0{sfx}").detach().float().cuda().requires_grad_(True)
                       for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
    Kp = (K + 7) // 8 * 8
    x_tm = torch.zeros((T, S, Kp), device="cuda")
    x_tm[:, :, :K] = x.transpose(0, 1).cuda()
    x_tm.requires_grad_(True)
    seq, last = f32.Lstm32Fn.apply(x_tm, lens.to(torch.int32).cuda() if ragged else None, True, *params)
    assert rel(seq, ref_seq) < 1e-4 and rel(last, ref_last) < 1e-4, (rel(seq, ref_seq), rel(last, ref_last))
    ((seq * w_seq.float().cuda()).sum() + (last * w_last.float().cuda()).sum()).backward()
    assert rel(x_tm.grad[:, :, :K].transpose(0, 1), xr.grad) < 1e-4, rel(x_tm.grad[:, :, :K].transpose(0, 1), xr.grad)
    i = 0
    for m in refs:
        for sfx in ("", "_reverse"):
            for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                e = rel(params[i].grad, getattr(m, f"{n}_l0{sfx}").grad)
                assert e < 1e-4, (n + sfx, e)
                i += 1


# ------------------------------------------------------------------------------------------------- whole model, fp32 mode
TOL32 = 1e-4


@pytest.fixture()
def fp32_mode():
    import dualvgr_videoqa_b200.autograd as ag
    ag.ACT[0] = F32
    yield
    ag.ACT[0] = BF16


def _build(cfg, training=True):
    from test_model_gpu import build
    model, inputs, ans = build(cfg, training)
    model.set_precision("fp32")
    return model, inputs, ans


@pytest.mark.parametrize("name", ["g1_B4_N8_U2", "g2_B3_N20_U3", "g3_B5_N16_U1", "g4_B16_N20_U3"])
def test_fp32_mode_against_reference_golden(golden, fp32_mode, name):
    """fp32 mode against the UNMODIFIED reference's float64 run (tests/golden): logits (eval and train), the unit stack's
    embeddings and graph outputs, the losses and the CE gradient at north_star's 1e-4; argmax identical on every row.
    The full-loss gradient is reported next to the reference's own fp32-vs-fp64 gap (the auxiliary terms are
    ill-conditioned: the reference's fp32 run itself misses its float64 run there) and gated by it."""
    import numpy as np
    from test_model_gpu import _probe, total_loss
    g = golden(name)
    cfg = [int(x) for x in g["cfg"]]
    N = cfg[1]
    model, inputs, ans = _build(cfg, training=False)
    with torch.no_grad():
        logits_eval = model(*inputs)[0]
    assert logits_eval.dtype == F32 and rel(logits_eval, g["f64_logits_eval"]) < TOL32, rel(logits_eval, g["f64_logits_eval"])
    model, inputs, ans = _build(cfg, training=True)
    out = model(*inputs)
    ref_logits = g["f64_logits_train"]
    e_log = rel(out[0], ref_logits)
    assert e_log < TOL32, e_log
    assert np.array_equal(out[0].argmax(1).cpu().numpy(), ref_logits.argmax(1))
    rows = g["embed_rows"] if "embed_rows" in g.files else slice(None)     # g4 keeps a seeded subset of the batch
    assert rel(out[1][rows], g["f64_aq_embed"]) < TOL32 and rel(out[2][rows], g["f64_mq_embed"]) < TOL32
    if "f64_com_app_0" in g.files:
        for i in range(len(out[3])):
            for key, lst in (("com_app", out[3]), ("com_mot", out[4]), ("aq_fusion", out[5]), ("mq_fusion", out[6])):
                assert lst[i].dtype == F32 and rel(lst[i], g[f"f64_{key}_{i}"]) < TOL32, (key, i)
    total, ce, com, dep = total_loss(out, ans, N)
    ref_total, ref_ce, ref_com, ref_dep = g["f64_losses"]
    f32_total, f32_ce, f32_com, f32_dep = g["f32_losses"]
    assert abs(float(ce) - ref_ce) < TOL32 * abs(ref_ce)
    assert abs(float(com) - ref_com) < max(4 * abs(f32_com - ref_com), 1e-3 * abs(ref_com))
    assert abs(float(dep) - ref_dep) < max(4 * abs(f32_dep - ref_dep), 1e-3 * abs(ref_dep))
    names = [str(n) for n in g["grad_names"]]
    params = dict(model.named_parameters())
    grads = torch.autograd.grad(ce, [params[n] for n in names], retain_graph=True, allow_unused=True)
    got_norm = np.array([0.0 if gr is None else float(gr.double().norm()) for gr in grads])
    got_proj = np.array([0.0 if gr is None else float((gr.double().cpu() * _probe(n, gr.shape)).sum())
                         for n, gr in zip(names, grads)])
    ref = g["f64_grad_ce"]
    e_norm = np.linalg.norm(got_norm - ref[:, 0]) / np.linalg.norm(ref[:, 0])
    e_proj = np.linalg.norm(got_proj - ref[:, 1]) / np.linalg.norm(ref[:, 1])
    floor_norm = np.linalg.norm(g["f32_grad_ce"][:, 0] - ref[:, 0]) / np.linalg.norm(ref[:, 0])
    grads_f = torch.autograd.grad(total, [params[n] for n in names], allow_unused=True)
    got_f = np.array([0.0 if gr is None else float(gr.double().norm()) for gr in grads_f])
    ref_f = g["f64_grad_full"]
    floor32 = np.linalg.norm(g["f32_grad_full"][:, 0] - ref_f[:, 0]) / np.linalg.norm(ref_f[:, 0])
    err_f = np.linalg.norm(got_f - ref_f[:, 0]) / np.linalg.norm(ref_f[:, 0])
    print(f"{name} fp32 mode vs reference fp64: logits {e_log:.2e}; CE-gradient norm vector {e_norm:.2e} (reference fp32 "
          f"{floor_norm:.2e}), probe projections {e_proj:.2e}; full-loss gradient {err_f:.2e} (reference fp32 {floor32:.2e})")
    assert e_norm < TOL32 and e_proj < 10 * TOL32
    # the auxiliary terms amplify a perturbation of the graph outputs by 10^2 - 10^3 (the reference's own fp32 run, whose
    # products are good to 1e-7, lands `floor32` away from its float64 run); fp32 mode's split products are good to ~2e-5
    assert err_f < max(TOL32, 4 * floor32, 1e-3), (err_f, floor32)


@pytest.mark.parametrize("cfg", [(6, 20, 8, 32, 60, 3), (24, 8, 8, 32, 60, 2), (8, 16, 8, 4002, 60, 1), (4, 64, 8, 50, 60, 1)])
def test_fp32_mode_full_gradient_tensors_against_oracle(fp32_mode, cfg):
    """Every parameter's full CE-gradient tensor against the oracle's float64 autograd: global relative L2 < 1e-4."""
    B, N, L, A, V, U = cfg
    model, inputs, ans = _build(cfg, training=True)
    out = model(*inputs)
    ce = torch.nn.functional.cross_entropy(out[0], ans)
    names = [n for n, _ in model.named_parameters()]
    grads = torch.autograd.grad(ce, [p for _, p in model.named_parameters()], allow_unused=True)
    sd = orc.cast_state_dict(orc.make_state_dict(U, A, V), torch.float64)
    for v in sd.values():
        if v.is_floating_point():
            v.requires_grad_(True)
    app, mot, q, qlen, ans_c = orc.make_inputs(B, N, L, A, V)
    ref_out = orc.dualvgr_forward(sd, U, app.double(), mot.double(), q, qlen, training=True)
    ref_ce = torch.nn.functional.cross_entropy(ref_out[0], ans_c)
    ref_grads = torch.autograd.grad(ref_ce, [sd[n] for n in names], allow_unused=True)
    assert rel(out[0], ref_out[0]) < TOL32, rel(out[0], ref_out[0])
    num = den = 0.0
    worst = []
    for n, gr, rg in zip(names, grads, ref_grads):
        if rg is None:
            continue
        gr = torch.zeros_like(rg) if gr is None else gr.double().cpu()
        num += float((gr - rg).pow(2).sum()); den += float(rg.pow(2).sum())
        worst.append((float((gr - rg).norm() / rg.norm().clamp_min(1e-30)), float(rg.norm()), n))
    print(f"fp32 mode, cfg {cfg}: global CE-gradient rel-L2 vs oracle fp64 {(num / den) ** 0.5:.2e}; logits "
          f"{rel(out[0], ref_out[0]):.2e}; worst tensors {sorted(worst)[-3:]}")
    assert (num / den) ** 0.5 < TOL32, sorted(worst)[-5:]


def test_fp32_mode_engine_step_matches_torch_adam(fp32_mode):
    """One TrainEngine step in fp32 mode (full loss, clip 12, Adam) against the oracle's float64 step on the same batch:
    loss at 1e-4, updated weights within 1e-4 of the step size."""
    import dualvgr_videoqa_b200.engine as E
    cfg = (8, 8, 8, 32, 60, 2)
    B, N, L, A, V, U = cfg
    model, inputs, ans = _build(cfg, training=True)
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    eng = E.TrainEngine(model, lr=1e-4)
    total = eng.train_step(*inputs, ans)
    sd = orc.cast_state_dict(orc.make_state_dict(U, A, V), torch.float64)
    ps = {k: v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running_" not in k}
    app, mot, q, qlen, ans_c = orc.make_inputs(B, N, L, A, V)
    ro = orc.dualvgr_forward(sd, U, app.double(), mot.double(), q, qlen, training=True)
    loss = torch.nn.functional.cross_entropy(ro[0], ans_c)
    com = sum(orc.common_loss(ro[3][i], ro[4][i]) for i in range(U))
    dep = sum(orc.loss_dependence(ro[5][i], ro[3][i], N) + orc.loss_dependence(ro[6][i], ro[4][i], N) for i in range(U))
    loss = loss + 1.0 * com / U + 1e-8 * dep / U
    opt = torch.optim.Adam(list(ps.values()), lr=1e-4)
    loss.backward()
    torch.nn.utils.clip_grad_norm_(list(ps.values()), 12.0)
    opt.step()
    assert abs(float(total) - float(loss)) < 1e-4 * abs(float(loss)), (float(total), float(loss))
    num = den = 0.0
    for n, p in model.named_parameters():
        step_ref = ps[n].detach() - before[n].double().cpu()
        step_got = p.detach().double().cpu() - before[n].double().cpu()
        num += float((step_got - step_ref).pow(2).sum()); den += float(step_ref.pow(2).sum())
    print(f"fp32 engine step: loss {float(total):.6f} vs {float(loss):.6f}; update rel-L2 {(num / den) ** 0.5:.2e}")
    assert (num / den) ** 0.5 < 2e-2        # Adam's first step is sign(g) * lr: only sign flips of ~zero gradients differ
    eng.close()


def test_fp32_gat_head_split_matches_whole_graph_launch(ops):
    """fp32 graph attention at a node count whose whole-graph tiles do not fit shared memory (N = 40: head-split launches, one
    virtual single-head graph per head) against the float64 formula: forward and every gradient at 1e-5; with dropout ON the
    keep rate of the output mask must be 1 - p for both launch shapes (the slices index the real graph's mask streams)."""
    import dualvgr_videoqa_b200.autograd as ag
    B, D, heads = 3, 768, 4
    Dh = D // heads
    for N, p_drop in ((40, 0.0), (40, 0.15), (20, 0.15)):
        g = torch.Generator().manual_seed(N)
        wh = torch.randn((B * N, D), generator=g).cuda()
        gate = torch.rand((B, N), generator=g).cuda()
        avec = (torch.randn((heads, 2 * Dh + 1), generator=g) * 0.1).cuda()
        adj = torch.full((N, N), 1.0 / N).cuda()
        dout = torch.randn((B * N, D), generator=g).cuda()
        outs, _ = ops.gat_attn_fwd([wh], [gate], [avec], adj, B, N, heads=heads, p_att=p_drop, p_out=p_drop, seed=77, streams=[5])
        out = outs[0]
        dwhs, dgates, davecs = ops.gat_attn_bwd([wh], [gate], [avec], [out], [dout], adj, B, N, heads=heads, p_att=p_drop,
                                                p_out=p_drop, seed=77, streams=[5])
        if p_drop == 0.0:
            whd = wh.double().cpu().view(B, N, heads, Dh).requires_grad_(True)
            gd, ad = gate.double().cpu().requires_grad_(True), avec.double().cpu().requires_grad_(True)
            s = (whd * ad[:, :Dh]).sum(-1)                      # [B, N, heads]
            t = (whd * ad[:, Dh:2 * Dh]).sum(-1)
            e = torch.nn.functional.leaky_relu(s[:, :, None, :] + t[:, None, :, :] + ad[:, 2 * Dh], 0.01)   # [B, i, j, heads]
            P = torch.softmax(e, dim=2)
            agg = torch.einsum("bijk,bjkc->bikc", P, whd * gd[:, :, None, None])
            ref = torch.nn.functional.elu(agg).reshape(B * N, D)
            assert rel(out, ref) < 1e-5, rel(out, ref)
            ref.backward(dout.double().cpu())
            assert rel(dwhs[0], whd.grad.reshape(B * N, D)) < 1e-5
            assert rel(dgates[0], gd.grad) < 1e-5
            assert rel(davecs[0], ad.grad) < 1e-5
        else:
            kept = float((out != 0).float().mean())
            assert abs(kept - (1 - p_drop)) < 0.02, kept
            if N == 40:
                first20 = out.view(B, N, heads, Dh)[0, :, :, :]
                assert bool(torch.isfinite(out).all()) and float(first20.abs().sum()) > 0
