"""torch.autograd.Function wrappers: each pairs a forward and a backward entry point of the C ABI so that the nn.Module
mirror in ``model/`` trains through ``loss.backward()`` exactly like the reference. PyTorch only routes tensors here
(allocation, views, concatenation of tiny parameter vectors); all arithmetic of the hot path is in the library."""
import collections
import os
import weakref

import torch
from torch.autograd import Function

from . import ops

BF16, F32 = torch.bfloat16, torch.float32

# activation dtype of the model mirror: bf16 (default, the fast path) or fp32 (DualVGR.set_precision("fp32"): fp32_path.py).
# The Functions below dispatch on the dtype of the tensors they are given; module code casts its inputs to ACT[0].
ACT = [BF16]

# ---------------------------------------------------------------------------------------------------------------------
# dropout bookkeeping: one seed per forward pass, one stream id per dropout site (regenerated, never stored)
# ---------------------------------------------------------------------------------------------------------------------
_rng = {"seed": 0x5EED, "site": 0, "epoch": 0}


def set_rank_seed(rank):
    """Data-parallel ranks draw independent dropout masks (the engine calls this after the weights are synchronised)."""
    _rng["rank"] = int(rank)


def begin_forward():
    """Called by DualVGR.forward: new seed for this pass, site counter reset."""
    _rng["seed"] = (int(torch.initial_seed()) * 1000003 + _rng["epoch"] * 7919 + 12345
                    + _rng.get("rank", 0) * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF
    _rng["epoch"] += 1
    _rng["site"] = 0


def _site(n=1):
    s = _rng["site"]
    _rng["site"] += n
    return _rng["seed"], s


# ---------------------------------------------------------------------------------------------------------------------
# bf16 operand cache for fp32 parameters (re-cast only when the parameter changed)
# ---------------------------------------------------------------------------------------------------------------------
_wcache = {}
_wepoch = [0]
# optional CUDA-event instrumentation of the dominant kernel (bench.py sets PROFILE["wih_gemm"] = [] to collect)
PROFILE = {}


# whole-sequence fused LSTM forward (dvgr_lstm_seq_fwd) instead of W_ih GEMM + T step launches; DVGR_LSTM_SEQ=0 keeps the
# two-kernel path (A/B measurements). SYNC_WORDS collects the kernels' sync buffers (last word = sticky timeout flag) of the
# most recent forward passes so that tests / bench can assert the dependency protocol never timed out.
LSTM_SEQ = [os.environ.get("DVGR_LSTM_SEQ", "1") != "0"]
WHH_TRANSPOSED = [os.environ.get("DVGR_WHH_T", "1") != "0"]


class _SyncLog(collections.deque):
    """Sync buffers of the recent whole-sequence LSTM launches; the current step's sticky error words are also collected for
    the engine's end-of-step check (ops.finalize_loss turns the loss into NaN if any is set)."""

    def append(self, sync):
        super().append(sync)
        _STEP_FLAGS.append(sync[-1:])


_STEP_FLAGS = []
SYNC_WORDS = _SyncLog(maxlen=16)


def begin_step_flags():
    del _STEP_FLAGS[:]


def step_flags():
    return list(_STEP_FLAGS[-16:])


def lstm_seq_timeouts():
    """Number of dependency-poll timeouts recorded by the recent whole-sequence LSTM launches (must be 0)."""
    return sum(int(w[-1].item()) for w in SYNC_WORDS)


def invalidate_weight_cache():
    """The flat-buffer optimizer updates parameters behind autograd's version counters: it calls this after a step."""
    _wepoch[0] += 1


def _versions(params):
    return tuple((p.data_ptr(), p._version) for p in params) + (_wepoch[0],)


# bf16 shadow of the engine's flat parameter buffer: {id(param): (weakref, bf16 view)}; kept current by the fused Adam kernel
SHADOW = {}


def _shadow_rows(params, out_cols, lstm_H):
    if lstm_H or not SHADOW:
        return None
    C = params[0].shape[1]
    if out_cols not in (None, C):
        return None
    ent = SHADOW.get(id(params[0]))
    if ent is None or ent[0]() is not params[0]:
        return None
    ptr, rows = ent[1].data_ptr(), 0
    for p in params:
        e = SHADOW.get(id(p))
        if e is None or e[0]() is not p or e[1].data_ptr() != ptr or p.shape[1] != C:
            return None
        ptr += p.numel() * 2
        rows += p.shape[0]
    return torch.as_strided(ent[1], (rows, C), (C, 1))


def bf16_rows(params, out_cols=None, lstm_H=0, tag=""):
    """bf16 operand made of the row-wise concatenation of fp32 matrices `params` (all [r_i, C]).
    Cached per parameter OBJECT (weak references: a freed model whose storage address is recycled by the caching
    allocator must not alias a live one) and re-cast whenever a version counter, data pointer or the optimizer epoch moves."""
    sh = _shadow_rows(params, out_cols, lstm_H)
    if sh is not None:
        return sh
    key = (tag, tuple(id(p) for p in params), out_cols, lstm_H)
    ver = _versions(params)
    ent = _wcache.get(key)
    if ent is not None and ent[0] == ver and all(r() is p for r, p in zip(ent[2], params)):
        return ent[1]
    C = params[0].shape[1]
    oc = out_cols or C
    rows = sum(p.shape[0] for p in params)
    buf = torch.empty((rows, oc), dtype=BF16, device=params[0].device)
    with torch.no_grad():       # ONE launch per 8 matrices (the per-step re-cast of the LSTM operands, outside the bf16 shadow)
        r = 0
        for i in range(0, len(params), 8):
            grp = [p.detach() for p in params[i:i + 8]]
            n = sum(p.shape[0] for p in grp)
            if len(grp) == 1:
                ops.cast_rows(grp[0], out=buf[r:r + n], out_cols=oc, lstm_H=lstm_H)
            else:
                ops.cast_rows_grouped(grp, buf[r:r + n], out_cols=oc, lstm_H=lstm_H)
            r += n
    if len(_wcache) > 4096:
        _wcache.clear()
    _wcache[key] = (ver, buf, tuple(weakref.ref(p) for p in params))
    return buf


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# ---------------------------------------------------------------------------------------------------------------------
# direct gradient accumulation (engine mode): when the parameters' .grad are pre-bound views of the engine's flat fp32
# gradient buffer, weight-gradient GEMMs add into them directly (split-K, fp32 atomics) and bias column-sums accumulate in
# place; the Function then returns None for that gradient, so autograd launches no separate accumulation kernel.
# ---------------------------------------------------------------------------------------------------------------------
DIRECT_GRAD = [False]
DIRECT_STATS = {"hits": 0, "misses": 0}


def grad_target(params):
    """[sum rows, cols] fp32 view over the .grad of `params` if they are bound, fp32, and contiguous in this order."""
    if not DIRECT_GRAD[0]:
        return None
    g0 = getattr(params[0], "grad", None)
    if g0 is None:
        DIRECT_STATS["misses"] += 1
        return None
    ptr, rows, cols = g0.data_ptr(), 0, params[0].shape[-1]
    for p in params:
        g = getattr(p, "grad", None)
        if g is None or g.dtype != F32 or not g.is_contiguous() or g.data_ptr() != ptr or p.shape[-1] != cols:
            DIRECT_STATS["misses"] += 1
            return None
        ptr += g.numel() * 4
        rows += g.numel() // cols
    DIRECT_STATS["hits"] += 1
    return torch.as_strided(g0, (rows, cols), (cols, 1))


def grad_groups(model):
    """Parameter groups that the fused kernels treat as ONE row-concatenated matrix; the engine lays each group out
    contiguously in its flat buffers so that grad_target() can hand the whole block to a single weight-gradient GEMM."""
    groups = []
    app = getattr(model, "visual_appearance_input_unit", None)
    if app is not None:
        e = app.encoder
        groups += [[e.weight_ih_l0, e.weight_ih_l0_reverse], [e.weight_hh_l0, e.weight_hh_l0_reverse]]
    lin = getattr(model, "linguistic_input_unit", None)
    if lin is not None:
        r, e = lin.concatRNN.rnn, lin.encoder
        groups += [[r.weight_ih_l0, r.weight_ih_l0_reverse, e.weight_ih_l0, e.weight_ih_l0_reverse],
                   [r.weight_hh_l0, r.weight_hh_l0_reverse, e.weight_hh_l0, e.weight_hh_l0_reverse]]
    unit = getattr(model, "visual_input_unit", None)
    if unit is not None and hasattr(unit, "acGCN"):
        for i in range(unit.layers):
            # the four graphs of a layer project through ONE batched GEMM [4][D][D] (fused_stack.UnitStackFn); its two view
            # attention projections through another [2][D][D]; the two cycle-query projections read the same input
            gats = (unit.acGCN[i], unit.appearance_GCN[i], unit.mcGCN[i], unit.motion_GCN[i])
            groups.append([att.W.weight for g in gats for att in g.attentions])
            groups.append([unit.attention_appearance[i].project[0].weight, unit.attention_motion[i].project[0].weight])
            qa, qm = unit.queryPunish_appear[i].query_weight, unit.queryPunish_motion[i].query_weight
            groups += [[qa.weight, qm.weight], [qa.bias, qm.bias]]
            groups.append([att.W.bias for g in gats for att in g.attentions])       # head biases: one column sum per graph
    return groups


# ---------------------------------------------------------------------------------------------------------------------
class LinearFn(Function):
    """y = act(x W^T + b) on the tcgen05 GEMM; backward = activation', dgrad (W read MN-major), wgrad, bias column-sum.
    x: [..., K'] bf16 with K' >= K (zero padded to a multiple of 8); W fp32 [N, K]; output bf16 (or fp32: the logits)."""

    @staticmethod
    def forward(ctx, x, weight, bias, act, out_f32, act_grad_folded=False, out_slot=None, dx_slot=None):
        """out_slot: optional 1-tuple with a preallocated [M, N] output buffer (see AppearanceEncoderFn).
        dx_slot: optional (PairSlot, index): the input gradient is written into that half of a shared [2, M, K] buffer."""
        ctx.dx_slot = dx_slot
        Kp = x.shape[-1]
        x2 = _rows2d(x)
        w = bf16_rows([weight], out_cols=Kp)
        y = ops.linear_fwd(x2, w, bias=bias, act=act, out_dtype=F32 if out_f32 else BF16,
                           out=out_slot[0] if out_slot is not None else None)
        ysave = None
        if act not in (None, "none") and not act_grad_folded:
            ysave = y if y.dtype == BF16 else y.to(BF16)       # act' only needs the sign / bf16-level value of the output
        ctx.save_for_backward(x2, w, ysave)
        ctx.act, ctx.out_f32, ctx.lead, ctx.K, ctx.has_bias = act, out_f32, x.shape[:-1], weight.shape[1], bias is not None
        ctx.wparam, ctx.bparam = weight, bias
        return y.view(*x.shape[:-1], weight.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w, y = ctx.saved_tensors
        N = w.shape[0]
        M = x2.shape[0]
        if ctx.out_f32:      # fp32 gradient of an fp32 output -> zero-padded bf16 operand, one library pass
            d = ops.cast_rows(_c(dy.reshape(M, N)).float(), out_cols=(N + 7) // 8 * 8)
        else:
            # (a column slice of a wider gradient — torch.cat's backward — is a valid GEMM operand as it is: no copy)
            d = _rows2d(dy) if (dy.dim() == 2 and y is None and dy.dtype == BF16) else _c(dy.reshape(M, N))
            if d.dtype != BF16:
                d = d.to(BF16)
        if y is not None:
            d = ops.act_bwd(d, y, ctx.act)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            slot = None
            if ctx.dx_slot is not None:
                slot = ctx.dx_slot[0].take(ctx.dx_slot[1], M, w.shape[1], d.device)
            dx = ops.linear_dgrad(d, w, out=slot).view(*ctx.lead, w.shape[1])
        if ctx.needs_input_grad[1]:
            tgt = grad_target([ctx.wparam])
            if tgt is not None:
                ops.linear_wgrad(d, x2, out=tgt, atomic=True, rows=N, cols=ctx.K)
            else:
                dw = ops.linear_wgrad(d, x2)[:N, :ctx.K]
        if ctx.has_bias and ctx.needs_input_grad[2]:
            tgt = _bias_target(ctx.bparam)
            if tgt is not None:
                ops.colsum(d[:, :N], out=tgt, accumulate=True)
            else:
                db = ops.colsum(d)[:N]
        return dx, dw, db, None, None, None, None, None


class PairSlot:
    """[2, M, K] bf16 gradient buffer shared by the backward passes of two Functions whose input gradients the consumer wants
    adjacent in memory (the MFB's two projections feed the unit stack's stacked [2, M, D] layout: no stacking copy)."""

    def __init__(self):
        self.buf, self.used = None, 2

    def take(self, idx, M, K, device):
        if self.used >= 2 or self.buf is None or tuple(self.buf.shape[1:]) != (M, K):
            self.buf, self.used = torch.empty((2, M, K), dtype=BF16, device=device), 0
        self.used += 1
        return self.buf[idx]


def _rows2d(x):
    """[..., K] -> [rows, K] without a copy when the rows are regularly strided (a column slice of a wider buffer is a valid
    TMA operand as long as its row pitch is a multiple of 16 bytes)."""
    if x.dim() == 2 and x.stride(1) == 1 and x.stride(0) % 8 == 0 and x.data_ptr() % 16 == 0:
        return x
    return _c(x.reshape(-1, x.shape[-1]))


def _bias_target(b):
    if not DIRECT_GRAD[0]:
        return None
    g = getattr(b, "grad", None)
    if g is None or g.dtype != F32 or not g.is_contiguous():
        return None
    return g


class LinearCatFn(Function):
    """y = x [W1; W2]^T + [b1; b2]: two nn.Linear layers that read the same input as ONE GEMM (forward, dgrad and wgrad).
    Used for the two QueryPunish.query_weight projections of a unit (reference model/utils.py:100 called twice per layer,
    models.py:142-147): each is a 256 x 300 x 768 product, i.e. pure launch latency when run on its own."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2):
        Kp = x.shape[-1]
        x2 = _c(x.reshape(-1, Kp))
        w = bf16_rows([w1, w2], out_cols=Kp, tag="cat")
        bias = torch.cat([b1.detach(), b2.detach()])
        y = ops.linear_fwd(x2, w, bias=bias)
        ctx.save_for_backward(x2, w)
        ctx.params = (w1, b1, w2, b2)
        ctx.lead = x.shape[:-1]
        return y.view(*x.shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w = ctx.saved_tensors
        w1, b1, w2, b2 = ctx.params
        N1, N2, K = w1.shape[0], w2.shape[0], w1.shape[1]
        d = _c(dy.reshape(x2.shape[0], N1 + N2))
        if d.dtype != BF16:
            d = d.to(BF16)
        dx = ops.linear_dgrad(d, w).view(*ctx.lead, w.shape[1]) if ctx.needs_input_grad[0] else None
        dw1 = dw2 = db1 = db2 = None
        tgt = grad_target([w1, w2])
        if tgt is not None:
            ops.linear_wgrad(d, x2, out=tgt, atomic=True, rows=N1 + N2, cols=K)
        else:
            dw = ops.linear_wgrad(d, x2)[:N1 + N2, :K]
            dw1, dw2 = dw[:N1], dw[N1:]
        t1, t2 = _bias_target(b1), _bias_target(b2)
        if t1 is not None and t2 is not None and t2.data_ptr() == t1.data_ptr() + N1 * 4:
            ops.colsum(d, out=torch.as_strided(t1, (N1 + N2,), (1,)), accumulate=True)
        elif t1 is not None and t2 is not None:
            ops.colsum(d[:, :N1], out=t1, accumulate=True)
            ops.colsum(d[:, N1:], out=t2, accumulate=True)
        else:
            db = ops.colsum(d)
            db1, db2 = db[:N1], db[N1:]
        return dx, dw1, db1, dw2, db2


def linear_cat(x, w1, b1, w2, b2):
    if x.dtype == F32:
        from . import fp32_path
        return fp32_path.linear_cat32(x, w1, b1, w2, b2)
    return LinearCatFn.apply(x, w1, b1, w2, b2)


def _route_small(param, grad):
    """Inside an engine step: queue `grad` for accumulation into the bound .grad view of `param` (all such tiny gradients
    land in ONE scatter launch at flush time) and return None, so autograd launches no accumulation kernel for it.
    Everywhere else: return `grad` unchanged."""
    if ops.DEFER_WGRAD[0] and grad is not None and grad.dtype == F32:
        tgt = _bias_target(param)
        if tgt is not None and tgt.numel() == grad.numel():
            ops.small_grad_enqueue(tgt, grad if grad.is_contiguous() else grad.contiguous())
            return None
    return grad


def linear(x, weight, bias=None, act=None, out_f32=False, act_grad_folded=False, out=None, dx_slot=None):
    """act_grad_folded: the consumer's backward kernel already returns d(pre-activation) (view attention, MFB pair-sum,
    read-out fold act' into their own pass), so this backward must not apply act' again."""
    if x.dtype == F32:          # fp32 mode: 3 x bf16 split products (fp32_path.Linear32Fn); `out` slots are a bf16-path layout
        from . import fp32_path
        y = fp32_path.linear32(x, weight, bias, act, act_grad_folded)
        if out is not None:
            raise ValueError("preallocated output slots are not supported in fp32 mode")
        return y
    return LinearFn.apply(x, weight, bias, act, out_f32, act_grad_folded, (out,) if out is not None else None, dx_slot)


# ---------------------------------------------------------------------------------------------------------------------
class DropoutFn(Function):
    @staticmethod
    def forward(ctx, x, p):
        ctx.p = p
        ctx.seed, ctx.sid = _site()
        return ops.dropout_raw(_c(x), p, ctx.seed, ctx.sid).view_as(x)

    @staticmethod
    def backward(ctx, dy):
        return ops.dropout_raw(_c(dy), ctx.p, ctx.seed, ctx.sid).view_as(dy), None


def dropout(x, p, training):
    return DropoutFn.apply(x, p) if (training and p > 0) else x


# ---------------------------------------------------------------------------------------------------------------------
_UNMAP = {}


def _lstm_unmap(H, ndir, device):
    """row_map for gate-interleaved rows -> nn.LSTM row order: interleaved row d*4H + 4j + g -> d*4H + g*H + j.
    Built once per (H, ndir, device) on the host (a constant: no index arithmetic kernels inside the train step)."""
    key = (H, ndir, str(device))
    m = _UNMAP.get(key)
    if m is None:
        r = torch.arange(ndir * 4 * H)
        d, rr = r // (4 * H), r % (4 * H)
        m = (d * 4 * H + (rr % 4) * H + rr // 4).to(torch.int32).to(device)
        _UNMAP[key] = m
    return m


def _lstm_bias_grads(dg, bias_params, H):
    """Bias gradients of an LSTM encoder from the gate gradients dg [rows, D*4H] (gate-interleaved columns).
    bias_params: (b_ih, b_hh) per direction, flattened. Engine step: queued as grouped column sums that de-interleave
    straight into the bound .grad views (returns Nones); otherwise computed at once and returned in nn.LSTM order."""
    D = len(bias_params) // 2
    tg = [_bias_target(b) for b in bias_params]
    if ops.DEFER_WGRAD[0] and all(t is not None for t in tg):
        for d in range(D):
            ops.colsum_enqueue(dg[:, d * 4 * H:(d + 1) * 4 * H], tg[2 * d], perm_H=H, out2=tg[2 * d + 1])
        return [None] * (2 * D)
    db = ops.colsum(dg).view(D, H, 4).transpose(1, 2).reshape(D, 4 * H)
    return [db[i // 2] for i in range(2 * D)]


class AppearanceEncoderFn(Function):
    """VisualAppearanceEncoder.forward (reference model/Preprocessing.py:209-234): prologue pass, ONE tcgen05 GEMM for the
    input-to-hidden product of both directions (N = 8H), T fused recurrent steps, final dropout."""

    @staticmethod
    def forward(ctx, app, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, p_in, p_out, training, out_slot=None,
                rows=None, err=None):
        """out_slot: optional 1-tuple holding a preallocated [B*N, 2H] bf16 buffer for the result (the unit stack carries
        the appearance and motion streams as ONE [2, B*N, D] tensor: its producers write straight into the halves).
        rows: optional [B] int32 video rows; app is then a device-resident store [V, N, F, Dv] and the prologue reads the
        batch app[rows] from it (err: the store's sticky out-of-range word)."""
        _, N, T, Dv = app.shape
        B = app.shape[0] if rows is None else rows.numel()
        S, H = B * N, w_hh.shape[1]
        seed, sid = _site(2)
        p_x = p_in if training else 0.0
        if rows is None:
            xa = ops.prep_features(_c(app).view(S * T, Dv), T, True, True, p_x, seed, sid)
        else:
            xa = ops.prep_features_gather(app, rows, T, True, True, p_x, seed, sid, err)
        wih = _lstm_weight([w_ih, w_ih_r], H, "ih")
        whh = _lstm_weight([w_hh, w_hh_r], H, "hh").view(2, 4 * H, H)
        bias = ops.lstm_pack_bias([b_ih.detach(), b_ih_r.detach()], [b_hh.detach(), b_hh_r.detach()], H)
        dst = out_slot[0] if out_slot is not None else None
        rec = PROFILE.get("wih_gemm")
        if rec is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        if LSTM_SEQ[0]:
            # ONE persistent launch: input projection + all T recurrent steps (pre-activations never reach HBM)
            gates, h_hist, c_hist, h_last, _, sync = ops.lstm_seq_fwd(
                xa.view(T, S, Dv), wih, whh, bias, h_last=dst if (dst is not None and not (training and p_out > 0)) else None)
            SYNC_WORDS.append(sync)
        else:
            gates = ops.linear_fwd(xa, wih, bias=bias, bn=256).view(T, S, 8 * H)
        if rec is not None:
            ev1.record()
            rec.append((ev0, ev1))
        if not LSTM_SEQ[0]:
            h_hist, c_hist, h_last, _ = ops.lstm_fwd(gates, whh)
        out = h_last
        p_o = p_out if training else 0.0
        if p_o > 0:
            out = ops.dropout_raw(h_last, p_o, seed, sid + 1, out=dst)
        elif dst is not None and out.data_ptr() != dst.data_ptr():
            dst.copy_(out)
            out = dst
        ctx.save_for_backward(xa, whh, gates, h_hist, c_hist)
        ctx.cfg = (B, N, T, Dv, S, H, p_o, seed, sid)
        ctx.wih_params, ctx.whh_params = [w_ih, w_ih_r], [w_hh, w_hh_r]
        ctx.bias_params = (b_ih, b_hh, b_ih_r, b_hh_r)
        return out.view(B, N, 2 * H)

    @staticmethod
    def backward(ctx, dout):
        xa, whh, gates, h_hist, c_hist = ctx.saved_tensors
        B, N, T, Dv, S, H, p_o, seed, sid = ctx.cfg
        dh = _c(dout.reshape(S, 2 * H))
        if p_o > 0:
            dh = ops.dropout_raw(dh, p_o, seed, sid + 1)
        if LSTM_SEQ[0]:                                          # blocked activated gates in, standard-layout gradients out
            gates, sync = ops.lstm_bwd(gates, whh, h_hist, c_hist, dh, whole_sequence=True, max_ctas=ops._cap())
            SYNC_WORDS.append(sync)
        else:
            ops.lstm_bwd(gates, whh, h_hist, c_hist, dh)         # gates now holds d(pre-activation gates)
        dg = gates.view(T * S, 8 * H)
        unmap = _lstm_unmap(H, 2, dg.device)
        t_ih, t_hh = grad_target(ctx.wih_params), grad_target(ctx.whh_params)
        if t_ih is not None:
            # (measured, r2: dealing ONE tile per CTA so that the question encoder's backward chain interleaves on a higher-
            #  priority stream moves that chain inside this launch but does not shorten the step: SM-time is conserved)
            ops.linear_wgrad(dg, xa, out=t_ih, row_map=unmap, atomic=True, dynamic=True, max_ctas=ops._cap(1))   # long launch next to the question encoder's backward
            dwih = None
        else:
            dwih = ops.linear_wgrad(dg, xa, row_map=unmap, bn=256)  # [8H, Dv] fp32 in nn.LSTM row order
        dbs = _lstm_bias_grads(dg, ctx.bias_params, H)
        # dW_hh[d] = sum_s dgates[t_d(s)]^T h_hist[d][s]   (segmented MN-major reduction, both directions in one launch)
        kin = (S + 63) // 64
        dwhh = t_hh.view(2, 4 * H, H) if t_hh is not None else torch.empty((2, 4 * H, H), dtype=F32, device=dg.device)
        wbn, wks = ops.wgrad_split(4 * H, H, (T - 1) * kin * 64, batch=2) if t_hh is not None else (0, 0)
        # (the step-0 term is skipped: h_0 = 0, and its slot is not even initialised in the whole-sequence layout)
        s0 = 1 if LSTM_SEQ[0] else 0
        if WHH_TRANSPOSED[0]:
            # computed TRANSPOSED, dW_hh^T [H, 4H] = h^T dgates: the 4H side becomes the 256-wide tile dimension (36 tiles of
            # 128 x 256 instead of 72 of 128 x 128 — the narrow tiles are bound by the operand traffic from L2, not by the
            # tensor pipe), then one small permuted add un-interleaves the gates into nn.LSTM row order
            dwt = torch.zeros((2, H, 4 * H), dtype=F32, device=dg.device)
            ops.gemm(h_hist, 1, gates, 1, H, 4 * H, (T - s0) * kin * 64, dwt, ldc=4 * H, batch=2, c_batch=4 * H * H,
                     a_c2=[s0, s0], a_c2_step=[1, 1], a_c3=[0, 1], b_c0=[0, 4 * H], b_c2=[s0, T - 1 - s0], b_c2_step=[1, -1],
                     k_inner=kin, beta=2, bn=256, ksplit=4, dynamic=True, max_ctas=ops._cap(1))
            nat = dwt.view(2, H, H, 4).permute(0, 3, 2, 1).reshape(2, 4 * H, H)       # [d][k][4j+g] -> [d][g*H+j][k]
            if t_hh is not None:
                dwhh.add_(nat)
            else:
                dwhh = nat
        else:
            ops.gemm(gates, 1, h_hist, 1, 4 * H, H, (T - s0) * kin * 64, dwhh, ldc=H, batch=2, c_batch=4 * H * H,
                     row_map=_lstm_unmap(H, 1, dg.device), a_c0=[0, 4 * H], a_c2=[s0, T - 1 - s0], a_c2_step=[1, -1],
                     b_c2=[s0, s0], b_c2_step=[1, 1], b_c3=[0, 1], k_inner=kin, beta=2 if t_hh is not None else 0,
                     bn=wbn, ksplit=wks, dynamic=True, max_ctas=ops._cap(1))
        g_ih = (None, None) if dwih is None else (dwih[:4 * H], dwih[4 * H:])
        g_hh = (None, None) if t_hh is not None else (dwhh[0], dwhh[1])
        # b_ih, b_hh, b_ih_reverse, b_hh_reverse: both biases of a direction get the same gradient
        return (None, g_ih[0], g_hh[0], dbs[0], dbs[1], g_ih[1], g_hh[1], dbs[2], dbs[3], None, None, None, None, None, None)


def _lstm_weight(params, H, tag):
    return bf16_rows(params, lstm_H=H, tag="lstm_" + tag)


# ---------------------------------------------------------------------------------------------------------------------
class QuestionEncoderFn(Function):
    """Both question BiLSTMs of InputUnitLinguisticDynamic (reference model/Preprocessing.py:97-101,112-123) as ONE
    4-direction fused recurrence: directions 0/1 = concatRNN (per-token states, zero at padded positions like
    pad_packed_sequence), directions 2/3 = encoder (final states of the packed run). No packing, no host sync on
    question_len: padded steps are masked inside the cell epilogue.
    words fp32 [B, L, W] (= tanh(dropout(embedding))), qlen int32 [B]; params = the 8 tensors of concatRNN.rnn then the 8 of
    encoder, each in nn.LSTM order (w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r).
    Returns (dynamic_q [B, L, 2H] bf16, question_embedding [B, 2H] bf16)."""

    @staticmethod
    def forward(ctx, words, qlen, *params):
        B, L, W = words.shape
        H = params[1].shape[1]
        Wp = (W + 7) // 8 * 8
        x = torch.zeros((L, B, Wp), dtype=BF16, device=words.device)
        x[:, :, :W] = words.transpose(0, 1)
        w_ih = [params[0], params[4], params[8], params[12]]
        w_hh = [params[1], params[5], params[9], params[13]]
        wih = bf16_rows(w_ih, out_cols=Wp, lstm_H=H, tag="lstm_ih")
        whh = bf16_rows(w_hh, lstm_H=H, tag="lstm_hh").view(4, 4 * H, H)
        bias = torch.cat([(params[4 * d + 2] + params[4 * d + 3]).view(4, H).t().reshape(-1) for d in range(4)]).detach()
        if LSTM_SEQ[0]:
            gates, h_hist, c_hist, h_last, seq_out, sync = ops.lstm_seq_fwd(x, wih, whh, bias, seq_len=qlen, want_seq=True)
            SYNC_WORDS.append(sync)
        else:
            gates = ops.linear_fwd(x.view(L * B, Wp), wih, bias=bias).view(L, B, 16 * H)
            h_hist, c_hist, h_last, seq_out = ops.lstm_fwd(gates, whh, seq_len=qlen, want_seq=True)
        ctx.save_for_backward(x, wih, whh, gates, h_hist, c_hist, qlen)
        ctx.cfg = (B, L, W, Wp, H)
        ctx.wih_params, ctx.whh_params = w_ih, w_hh
        ctx.bias_params = [params[4 * d + j] for d in range(4) for j in (2, 3)]
        return seq_out[:, :, :2 * H].contiguous(), h_last[:, 2 * H:].contiguous()

    @staticmethod
    def backward(ctx, d_dq, d_q):
        x, wih, whh, gates, h_hist, c_hist, qlen = ctx.saved_tensors
        B, L, W, Wp, H = ctx.cfg
        dev = x.device
        dh_seq = torch.zeros((B, L, 4 * H), dtype=BF16, device=dev)
        dh_last = torch.zeros((B, 4 * H), dtype=BF16, device=dev)
        if d_dq is not None:
            dh_seq[:, :, :2 * H] = d_dq
        if d_q is not None:
            dh_last[:, 2 * H:] = d_q
        if LSTM_SEQ[0]:
            gates, sync = ops.lstm_bwd(gates, whh, h_hist, c_hist, dh_last, seq_len=qlen, dh_seq=dh_seq, whole_sequence=True)
            SYNC_WORDS.append(sync)
        else:
            ops.lstm_bwd(gates, whh, h_hist, c_hist, dh_last, seq_len=qlen, dh_seq=dh_seq)
        dg = gates.view(L * B, 16 * H)
        x2 = x.view(L * B, Wp)
        dwords = None
        if ctx.needs_input_grad[0]:
            dwords = ops.linear_dgrad(dg, wih).view(L, B, Wp)[:, :, :W].transpose(0, 1).float()
        unmap = _lstm_unmap(H, 4, dev)
        t_ih, t_hh = grad_target(ctx.wih_params), grad_target(ctx.whh_params)
        if t_ih is not None:
            ops.linear_wgrad(dg, x2, out=t_ih, row_map=unmap, atomic=True, cols=W)
            dwih = None
        else:
            dwih = ops.linear_wgrad(dg, x2, row_map=unmap)[:, :W]
        db = torch.empty(16 * H, dtype=F32, device=dev)
        db[unmap.long()] = ops.colsum(dg)
        kin = (B + 63) // 64
        dwhh = t_hh.view(4, 4 * H, H) if t_hh is not None else torch.empty((4, 4 * H, H), dtype=F32, device=dev)
        s0 = 1 if LSTM_SEQ[0] else 0        # the step-0 term is zero (h_0 = 0) and its slot uninitialised: skipped
        ops.gemm(gates, 1, h_hist, 1, 4 * H, H, (L - s0) * kin * 64, dwhh, ldc=H, batch=4, c_batch=4 * H * H,
                 row_map=_lstm_unmap(H, 1, dev), a_c0=[4 * H * d for d in range(4)], a_c2=[s0, L - 1 - s0, s0, L - 1 - s0],
                 a_c2_step=[1, -1, 1, -1], b_c2=[s0, s0, s0, s0], b_c2_step=[1, 1, 1, 1], b_c3=[0, 1, 2, 3], k_inner=kin,
                 beta=2 if t_hh is not None else 0)
        grads = []
        for d in range(4):
            sl = slice(4 * H * d, 4 * H * (d + 1))
            grads += [None if dwih is None else dwih[sl], None if t_hh is not None else dwhh[d],
                      _route_small(ctx.bias_params[2 * d], db[sl]), _route_small(ctx.bias_params[2 * d + 1], db[sl])]
        return (dwords, None) + tuple(grads)


# ---------------------------------------------------------------------------------------------------------------------
class QAttnFn(Function):
    """QueryAttn.forward after feat_enhance (reference model/utils.py:68-84). y [B,L,D] bf16, words [B,L,Wp] bf16
    (zero padded to Wp), qlen int32. Returns q_c [B, Wp] bf16 (zero padded) and alpha [B, L] fp32 (not differentiated)."""

    @staticmethod
    def forward(ctx, y, words, qlen, fc_w, fc_b, W):
        y, words = _c(y), _c(words)
        wf = _c(fc_w.detach().view(-1))
        qc, alpha, nrm, prob, ssum = ops.qattn_fwd(y, wf, fc_b.detach(), qlen, words, W, words.shape[-1])
        ctx.save_for_backward(y, words, qlen, wf, alpha, nrm, prob, ssum)
        ctx.W = W
        ctx.fc = (fc_w, fc_b)
        ctx.mark_non_differentiable(alpha)
        return qc, alpha

    @staticmethod
    def backward(ctx, dqc, _dalpha):
        y, words, qlen, wf, alpha, nrm, prob, ssum = ctx.saved_tensors
        dy, dwords, dwf, dcf = ops.qattn_bwd(_c(dqc), y, wf, qlen, words, ctx.W, alpha, nrm, prob, ssum)
        return dy, dwords, None, _route_small(ctx.fc[0], dwf.view(1, -1)), _route_small(ctx.fc[1], dcf.view(1)), None


class GateFn(Function):
    """QueryPunish gates of both streams (reference model/utils.py:101-103): g = sigmoid(X . query)."""

    @staticmethod
    def forward(ctx, xa, xm, query):
        xa, xm, query = _c(xa), _c(xm), _c(query)
        ga, gm = ops.gate_fwd(xa, xm, query)
        ctx.save_for_backward(xa, xm, query, ga, gm)
        return ga, gm

    @staticmethod
    def backward(ctx, dga, dgm):
        xa, xm, query, ga, gm = ctx.saved_tensors
        dxa, dxm = torch.zeros_like(xa), torch.zeros_like(xm)
        dq = ops.gate_bwd(xa, xm, query, ga, gm, _c(dga), None, _c(dgm), None, dxa, dxm)
        return dxa, dxm, dq


# ---------------------------------------------------------------------------------------------------------------------
class GatLayerFn(Function):
    """Several punishGATs in one shot (reference model/GraphNN.py:95-113,174-178): per input stream ONE batched projection
    GEMM for all graphs reading that stream, then ONE fused attention launch for all graphs (<= 4).
    A DualVGR unit calls it with 2 streams and graph_stream = (0, 0, 1, 1): acGCN, appearance_GCN, mcGCN, motion_GCN
    (reference model/models.py:151-158).
    tensors = xs (n_streams x [B,N,D] bf16) + gates (n_streams x [B,N] f32)
              + per graph, per head: W.weight, W.bias, a.weight, a.bias
    returns: per stream a stack [n_graphs_of_stream, B*N, D] bf16, then per graph a dense fp32 copy [B,N,D]."""

    @staticmethod
    def forward(ctx, graph_stream, adj, p, training, heads, *tensors):
        ns, G = max(graph_stream) + 1, len(graph_stream)
        xs, gates_in, params = tensors[:ns], tensors[ns:2 * ns], tensors[2 * ns:]
        B, N, D = xs[0].shape
        M, Dh = B * N, D // heads
        pdrop = p if training else 0.0
        seed, sid = _site(3 * G)          # graph g: input dropout sid+g, attention sid+G+2g, output sid+G+2g+1
        gp = [params[g * heads * 4:(g + 1) * heads * 4] for g in range(G)]
        of_stream = [[g for g in range(G) if graph_stream[g] == s] for s in range(ns)]
        # packed per-graph operands of the attention kernels: avec [heads][2Dh+1] = (a.weight | a.bias) per head, and the
        # concatenated head biases of each stream's projection GEMM — gathered from the parameters by ONE scatter launch
        avec_all = torch.empty((G, heads, 2 * Dh + 1), dtype=F32, device=xs[0].device)
        # train mode (every graph reads its own dropped copy of its stream) with the graphs listed stream by stream: ALL
        # graphs share ONE stacked set of buffers, so the projections of both streams are one batched GEMM (forward and
        # dgrad) — 480 tiles in 3.2 waves instead of two launches of 240 tiles in 2 waves each
        first = [of_stream[s][0] if of_stream[s] else 0 for s in range(ns)]
        stacked = (pdrop > 0 and G <= 4 and [g for s in range(ns) for g in of_stream[s]] == list(range(G)))
        bias_G = torch.empty((G, D), dtype=F32, device=xs[0].device)
        bias_all = [bias_G[first[s]:first[s] + len(of_stream[s])] for s in range(ns)]
        segs = []
        for g in range(G):
            for k in range(heads):
                segs.append((avec_all[g, k, :2 * Dh], gp[g][4 * k + 2].detach().reshape(-1)))
                segs.append((avec_all[g, k, 2 * Dh:], gp[g][4 * k + 3].detach().reshape(-1)))
        for s in range(ns):
            for i, g in enumerate(of_stream[s]):
                for k in range(heads):
                    segs.append((bias_all[s][i, k * Dh:(k + 1) * Dh], gp[g][4 * k + 1].detach()))
        ops.scatter(segs, False)
        avecs = [avec_all[g] for g in range(G)]
        whs, xts, wbufs, outs_s = [], [], [], []
        wh_list, out_list = [None] * G, [None] * G
        wb_all = None
        if stacked:
            dev0 = xs[0].device
            xt_all = torch.empty((G, M, D), dtype=BF16, device=dev0)
            wh_all = torch.empty((G, M, D), dtype=BF16, device=dev0)
            out_all = torch.empty((G, M, D), dtype=BF16, device=dev0)
            wb_all = bf16_rows([gp[g][4 * k] for g in range(G) for k in range(heads)], tag="gat_all").view(G, D, D)
        for s in range(ns):
            gs = of_stream[s]
            cnt = len(gs)
            x = _c(xs[s]).view(M, D)
            if stacked:
                g0 = first[s]
                for g in gs:
                    ops.dropout_raw(x, pdrop, seed, sid + g, out=xt_all[g])
                xt, wb, wh, out = xt_all[g0:g0 + cnt], wb_all[g0:g0 + cnt], wh_all[g0:g0 + cnt], out_all[g0:g0 + cnt]
            else:
                wb = bf16_rows([gp[g][4 * k] for g in gs for k in range(heads)], tag="gat").view(cnt, D, D)
                bias = bias_all[s]
                wh = torch.empty((cnt, M, D), dtype=BF16, device=x.device)
                if pdrop > 0:
                    xt = torch.stack([ops.dropout_raw(x, pdrop, seed, sid + g) for g in gs])
                    a_c2 = list(range(cnt))
                else:
                    xt, a_c2 = x, [0] * cnt
                ops.gemm(xt, 0, wb, 0, M, D, D, wh, ldc=D, bias=bias, batch=cnt, c_batch=M * D, bias_batch=D,
                         a_c2=a_c2, b_c2=list(range(cnt)))
                out = torch.empty((cnt, M, D), dtype=BF16, device=x.device)
            for i, g in enumerate(gs):
                wh_list[g], out_list[g] = wh[i], out[i]
            whs.append(wh); xts.append(xt); wbufs.append(wb); outs_s.append(out)
        if stacked:
            ops.gemm(xt_all, 0, wb_all, 0, M, D, D, wh_all, ldc=D, bias=bias_G, batch=G, c_batch=M * D, bias_batch=D,
                     a_c2=list(range(G)), b_c2=list(range(G)))
        streams = [sid + G + 2 * g for g in range(G)]
        gate_list = [_c(gates_in[graph_stream[g]]) for g in range(G)]
        _, f32s = ops.gat_attn_fwd(wh_list, gate_list, avecs, adj, B, N, heads=heads, p_att=pdrop, p_out=pdrop, seed=seed,
                                   streams=streams, outs=out_list, want_f32=True)
        ctx.save_for_backward(adj, *xts, *wbufs, *whs, *outs_s, *gate_list, *avecs)
        ctx.stacked_wb = wb_all                 # (bf16 operand cache entry, not an autograd tensor) stacked mode only
        ctx.cfg = (B, N, D, M, heads, pdrop, seed, sid, streams, graph_stream, of_stream)
        ctx.wparams = [[gp[g][4 * k] for g in of_stream[s] for k in range(heads)] for s in range(ns)]
        ctx.hparams = gp
        return tuple(outs_s) + tuple(f32s)

    @staticmethod
    def backward(ctx, *grads_out):
        B, N, D, M, heads, pdrop, seed, sid, streams, graph_stream, of_stream = ctx.cfg
        ns, G = len(of_stream), len(graph_stream)
        sv = ctx.saved_tensors
        adj = sv[0]
        xts, wbufs, whs, outs_s = sv[1:1 + ns], sv[1 + ns:1 + 2 * ns], sv[1 + 2 * ns:1 + 3 * ns], sv[1 + 3 * ns:1 + 4 * ns]
        gate_list = list(sv[1 + 4 * ns:1 + 4 * ns + G])
        avecs = list(sv[1 + 4 * ns + G:])
        Dh = D // heads
        dev = adj.device
        douts_s = [(_c(grads_out[s]) if grads_out[s] is not None else torch.zeros_like(outs_s[s])) for s in range(ns)]
        d32 = [None if t is None else _c(t) for t in grads_out[ns:ns + G]]
        wh_list, out_list, dout_list, dwh_list = [None] * G, [None] * G, [None] * G, [None] * G
        wb_all = ctx.stacked_wb
        stacked = wb_all is not None
        if stacked:
            dwh_all = torch.empty((G, M, D), dtype=BF16, device=dev)
            firsts = [of_stream[s][0] for s in range(ns)]
            dwh_s = [dwh_all[firsts[s]:firsts[s] + len(of_stream[s])] for s in range(ns)]
        else:
            dwh_s = [torch.empty_like(w) for w in whs]
        for s in range(ns):
            for i, g in enumerate(of_stream[s]):
                wh_list[g], out_list[g], dout_list[g], dwh_list[g] = whs[s][i], outs_s[s][i], douts_s[s][i], dwh_s[s][i]
        _, dgates, davecs = ops.gat_attn_bwd(wh_list, gate_list, avecs, out_list, dout_list, adj, B, N, heads=heads,
                                             p_att=pdrop, p_out=pdrop, seed=seed, streams=streams, douts32=d32,
                                             dwhs=dwh_list)
        dxs, dgs = [], []
        dW, db = [None] * G, [None] * G
        if stacked:      # one dgrad GEMM and one bias-gradient reduction for the graphs of BOTH streams
            dxt_all = torch.empty((G, M, D), dtype=BF16, device=dev)
            ops.gemm(dwh_all, 0, wb_all, 1, M, D, D, dxt_all, ldc=D, batch=G, c_batch=M * D, a_c2=list(range(G)),
                     b_c2=list(range(G)))
            dbs_all = ops.colsum_batched(dwh_all)
        for s in range(ns):
            gs = of_stream[s]
            cnt = len(gs)
            dwh, wb, xt = dwh_s[s], wbufs[s], xts[s]
            tgt = grad_target(ctx.wparams[s])
            direct = tgt is not None
            dWs = tgt.view(cnt, D, D) if direct else torch.empty((cnt, D, D), dtype=F32, device=dev)
            wbn, wks = ops.wgrad_split(D, D, M, batch=cnt) if direct else (0, 0)
            wkw = dict(beta=2, bn=wbn, ksplit=wks) if direct else {}
            if pdrop > 0:
                if stacked:
                    dxt = dxt_all[gs[0]:gs[0] + cnt]
                else:
                    dxt = torch.empty((cnt, M, D), dtype=BF16, device=dev)
                    ops.gemm(dwh, 0, wb, 1, M, D, D, dxt, ldc=D, batch=cnt, c_batch=M * D, a_c2=list(range(cnt)),
                             b_c2=list(range(cnt)))
                dx = ops.dropout_raw(dxt[0], pdrop, seed, sid + gs[0])
                for i in range(1, cnt):
                    ops.act_bwd(dxt[i], None, "none", out=dx, accumulate=True, p=pdrop, seed=seed, stream_id=sid + gs[i])
                if direct and ops.DEFER_WGRAD[0]:
                    for i in range(cnt):
                        ops.wgrad_enqueue(dwh[i], xt[i], dWs[i])
                else:
                    ops.gemm(dwh, 1, xt, 1, D, D, M, dWs, ldc=D, batch=cnt, c_batch=D * D, a_c2=list(range(cnt)),
                             b_c2=list(range(cnt)), **wkw)
            else:
                dx = ops.linear_dgrad(dwh[0], wb[0])
                for i in range(1, cnt):
                    ops.linear_dgrad(dwh[i], wb[i], out=dx, beta=True)
                if direct and ops.DEFER_WGRAD[0]:
                    for i in range(cnt):
                        ops.wgrad_enqueue(dwh[i], xt, dWs[i])
                else:
                    ops.gemm(dwh, 1, xt, 1, D, D, M, dWs, ldc=D, batch=cnt, c_batch=D * D, a_c2=list(range(cnt)),
                             b_c2=[0] * cnt, **wkw)
            dxs.append(dx.view(B, N, D))
            dg = dgates[gs[0]]
            for g in gs[1:]:
                dg = dg + dgates[g]
            dgs.append(dg)
            dbs = dbs_all[gs[0]:gs[0] + cnt] if stacked else ops.colsum_batched(dwh)      # head-bias gradients of the graphs
            for i, g in enumerate(gs):
                dW[g], db[g] = (None if direct else dWs[i]), dbs[i]
        grads = []
        small = []        # (bound .grad view, gradient) pairs of the per-head biases / attention vectors
        for g in range(G):
            for k in range(heads):
                hp = ctx.hparams[g][4 * k:4 * k + 4]                 # W.weight, W.bias, a.weight, a.bias of this head
                pieces = [db[g][k * Dh:(k + 1) * Dh], davecs[g][k, :2 * Dh].reshape(1, 2 * Dh), davecs[g][k, 2 * Dh:].reshape(1)]
                outs = []
                for prm, piece in zip(hp[1:], pieces):
                    tgt = _bias_target(prm)
                    if tgt is not None:
                        small.append((tgt, piece))
                        outs.append(None)
                    else:
                        outs.append(piece)
                grads += [None if dW[g] is None else dW[g][k * Dh:(k + 1) * Dh]] + outs
        ops.scatter_add(small)       # one launch for (up to) 48 tiny accumulations instead of one elementwise launch each
        return (None, None, None, None, None) + tuple(dxs) + tuple(dgs) + tuple(grads)


class ViewAttnFn(Function):
    """AttentionSFGCN tail + residual (reference model/Attention.py:21-23, model/models.py:168-169)."""

    @staticmethod
    def forward(ctx, hidden, z, x, w2):
        hidden, z, x = _c(hidden), _c(z), _c(x)
        w2v = _c(w2.detach().view(-1))
        x2 = x.view(-1, x.shape[-1])
        xnew, embed, beta = ops.view_attn_fwd(hidden, z, x2, w2v)
        ctx.save_for_backward(hidden, z, w2v, beta)
        ctx.w2 = w2
        return xnew.view_as(x), embed.view_as(x)

    @staticmethod
    def backward(ctx, dxnew, dembed):
        hidden, z, w2v, beta = ctx.saved_tensors
        D = z.shape[-1]
        if dxnew is None:
            dxnew = torch.zeros(z.shape[1:], dtype=z.dtype, device=z.device)
        dxn = _c(dxnew).view(-1, D)
        de = _c(dembed).view(-1, D) if dembed is not None else None
        dz, dhid, dw2 = ops.view_attn_bwd(dxn, de, hidden, z, w2v, beta)
        return dhid, dz, dxnew, _route_small(ctx.w2, dw2.view(1, -1))


class MfbPairFn(Function):
    """MFB product + pair-sum (reference model/fusions/fusions.py:433-441). Inputs are ELU outputs; the backward returns
    gradients w.r.t. the PRE-activations of linear0 / linear1 (ELU' folded in)."""

    @staticmethod
    def forward(ctx, x0, x1):
        x0, x1 = _c(x0), _c(x1)
        lead = x0.shape[:-1]
        a, b = x0.view(-1, x0.shape[-1]), x1.view(-1, x1.shape[-1])
        z = ops.mfb_fwd(a, b)
        ctx.save_for_backward(a, b)
        ctx.lead = lead
        return z.view(*lead, z.shape[-1])

    @staticmethod
    def backward(ctx, dz):
        a, b = ctx.saved_tensors
        d0, d1 = ops.mfb_bwd(_c(dz).view(-1, dz.shape[-1]), a, b)
        return d0.view(*ctx.lead, -1), d1.view(*ctx.lead, -1)


class ReadoutFn(Function):
    """ContextSelfAttn tail (reference model/AnswerDecoder.py:176-180). Backward returns d(pre-activation of v_proj) for u."""

    @staticmethod
    def forward(ctx, v, u, w, c):
        v, u = _c(v), _c(u)
        wv = _c(w.detach().view(-1))
        pooled, alpha = ops.readout_fwd(v, u, wv, c.detach())
        ctx.save_for_backward(v, u, wv, alpha)
        ctx.wc = (w, c)
        return pooled

    @staticmethod
    def backward(ctx, dp):
        v, u, wv, alpha = ctx.saved_tensors
        dpc = dp if (dp.dim() == 2 and dp.stride(1) == 1) else _c(dp)
        tw, tc = _bias_target(ctx.wc[0]), _bias_target(ctx.wc[1])
        if ops.DEFER_WGRAD[0] and tw is not None and tc is not None:
            # engine step: the two per-sample partial reductions ride the grouped column sum at the end of the step
            dv, du, dw_part, dc_part = ops.readout_bwd(dpc, v, u, wv, alpha, raw=True)
            ops.colsum_enqueue(dw_part, tw.view(-1))
            ops.colsum_enqueue(dc_part, tc.view(-1))
            return dv, du, None, None
        dv, du, dw, dc = ops.readout_bwd(dpc, v, u, wv, alpha)
        return dv, du, _route_small(ctx.wc[0], dw.view(1, -1)), _route_small(ctx.wc[1], dc.view(1))


class BatchNormFn(Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, run_mean, run_var, training, momentum, eps, sync=None):
        """sync = (process group, world size) -> synchronised BatchNorm: batch statistics over ALL ranks' rows (two tiny
        all-reduces per step); None -> statistics of this rank's rows (standard DDP)."""
        x = _c(x)
        ext, Btot = None, x.shape[0]
        if training and sync is not None:
            import torch.distributed as dist
            ext = ops.bn_stats(x)
            dist.all_reduce(ext, op=dist.ReduceOp.SUM, group=sync[0])
            Btot = x.shape[0] * sync[1]
        y, mean, rstd = ops.bn_fwd(x, gamma.detach(), beta.detach(), run_mean, run_var, training, momentum, eps, ext, Btot,
                                   out_dtype=ACT[0])
        ctx.save_for_backward(x, gamma.detach(), mean, rstd)
        ctx.training = training
        ctx.affine = (gamma, beta)
        ctx.sync = sync if (training and sync is not None) else None
        ctx.Btot = Btot
        ctx.ydt = y.dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, mean, rstd = ctx.saved_tensors
        dy = _c(dy)
        if dy.dtype != ctx.ydt:
            dy = dy.to(ctx.ydt)
        if ctx.sync is not None:
            import torch.distributed as dist
            _, dg, db = ops.bn_bwd(dy, x, gamma, mean, rstd, True, stats_only=True)      # LOCAL sums = this rank's dgamma / dbeta
            sums = torch.stack([db, dg])
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=ctx.sync[0])
            dx, _, _ = ops.bn_bwd(dy, x, gamma, mean, rstd, True, ext_sums=sums, Btot=ctx.Btot)
        else:
            dx, dg, db = ops.bn_bwd(dy, x, gamma, mean, rstd, ctx.training)
        return dx, _route_small(ctx.affine[0], dg), _route_small(ctx.affine[1], db), None, None, None, None, None, None


class CrossEntropyFn(Function):
    """Mean cross-entropy with the gradient produced in the same launch."""

    @staticmethod
    def forward(ctx, logits, answers, unit_grad=False):
        """unit_grad: the caller back-propagates the returned loss with coefficient exactly 1 (the engine), so backward hands
        the stored gradient on as it is."""
        loss, dlog, correct = ops.cross_entropy(_c(logits), answers, grad_f32=True)
        ctx.save_for_backward(dlog)
        ctx.unit_grad = bool(unit_grad)
        ctx.mark_non_differentiable(correct)
        return loss, correct

    @staticmethod
    def backward(ctx, g, _):
        (dlog,) = ctx.saved_tensors
        return (dlog if ctx.unit_grad else dlog * g), None, None


class AuxLossFn(Function):
    """The three auxiliary-loss pairs of one DualVGR unit (reference train.py:148-154, utils.py:10-31) in ONE fused call:
    coef_com * sum (G_ca - G_cm)^2 + coef_dep * (HSIC(aq, ca) + HSIC(mq, cm)), value and all four gradients together.
    Returns (combined scalar, [3] tensor of the coef-scaled terms (not differentiated))."""

    @staticmethod
    def forward(ctx, ca, cm, aq, mq, coef_com, coef_dep, unit_grad=False):
        """unit_grad: the caller adds the returned scalar to its total loss with coefficient exactly 1 (train.py:154 with
        alpha / beta already folded into the coefficients), so backward returns the stored gradients as they are instead
        of launching four [B,N,D] multiplications by a scalar that is 1."""
        ctx.unit_grad = bool(unit_grad)
        ca, cm, aq, mq = (_c(t.float()) for t in (ca, cm, aq, mq))
        vals, (d_ca, d_cm, d_aq, d_mq) = ops.aux_loss_unit(ca, cm, aq, mq, coef_com, coef_dep, precise=ACT[0] == F32)
        ctx.save_for_backward(d_ca, d_cm, d_aq, d_mq)
        ctx.mark_non_differentiable(vals)
        return vals.sum(), vals

    @staticmethod
    def backward(ctx, g, _):
        d_ca, d_cm, d_aq, d_mq = ctx.saved_tensors
        if ctx.unit_grad:
            return d_ca, d_cm, d_aq, d_mq, None, None, None
        return d_ca * g, d_cm * g, d_aq * g, d_mq * g, None, None, None


class PairLossFn(Function):
    """common_loss / loss_dependence (reference utils.py:10-31): value and gradients from one fused launch."""

    @staticmethod
    def forward(ctx, x, y, mode, coef):
        loss, dx, dy = ops.pair_loss(_c(x.float()), _c(y.float()), mode, coef)
        ctx.save_for_backward(dx, dy)
        return loss

    @staticmethod
    def backward(ctx, g):
        dx, dy = ctx.saved_tensors
        return dx * g, dy * g, None, None
