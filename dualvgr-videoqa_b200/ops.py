"""Functional layer over the C ABI: every function takes torch CUDA tensors, allocates outputs with torch (device
memory and streams are torch's), and launches the library's kernels on the current stream.

No arithmetic of the hot path happens in PyTorch here; there is no fallback if the library is missing."""
import ctypes
import os

import torch

from . import _lib

ACT_NONE, ACT_ELU, ACT_TANH = 0, 1, 2
BF16, F32 = torch.bfloat16, torch.float32
_ACT = {None: 0, "none": 0, "elu": 1, "tanh": 2}


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _check_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.DvgrError("dualvgr_b200 ops need CUDA tensors: there is no CPU path")


def operand(t, major):
    """Describe a tensor whose LAST dim is contiguous as a GEMM operand. major 0: K-major (rows x K), 1: MN-major (K x rows).
    Leading dims (up to 2) become outer TMA dims 2, 3."""
    assert t.dtype == torch.bfloat16 and t.stride(-1) == 1 and 2 <= t.dim() <= 4
    op = _lib.Operand()
    op.ptr = t.data_ptr()
    op.major = major
    op.ndim = t.dim()
    shape = list(t.shape)[::-1]
    strides = list(t.stride())[::-1]
    for i in range(t.dim()):
        op.dims[i] = shape[i]
        op.strides[i] = strides[i]
    return op


def gemm(A, a_major, B, b_major, M, N, K, C, *, ldc=None, bias=None, act=None, beta=False, batch=1, c_batch=0,
         bias_batch=0, row_map=None, a_c0=None, a_c2=None, a_c3=None, b_c0=None, b_c2=None, b_c3=None, k_inner=0,
         a_c2_step=None, b_c2_step=None, bn=0, max_ctas=0, ksplit=0, dynamic=False):
    """Raw tcgen05 GEMM: C[b][m][n] = act(sum_k A*B + bias) (+C). dynamic: CTAs claim tiles from a (freshly zeroed) device
    counter instead of the static round-robin deal — for long launches that overlap kernels on other streams."""
    _check_cuda(A, B, C, bias)
    args = _lib.GemmArgs()
    args.A = operand(A, a_major)
    args.B = operand(B, b_major)
    args.M, args.N, args.K, args.batch = M, N, K, batch
    for name, val in (("a_c0", a_c0), ("a_c2", a_c2), ("a_c3", a_c3), ("b_c0", b_c0), ("b_c2", b_c2), ("b_c3", b_c3),
                      ("a_c2_step", a_c2_step), ("b_c2_step", b_c2_step)):
        if val is not None:
            arr = getattr(args, name)
            for i, v in enumerate(val):
                arr[i] = int(v)
    args.k_inner = k_inner
    args.C = C.data_ptr()
    args.ldc = ldc if ldc is not None else C.stride(-2)
    args.c_batch = c_batch
    assert C.dtype in (torch.float32, torch.bfloat16)
    args.out_f32 = 1 if C.dtype == torch.float32 else 0
    args.act = _ACT[act] if not isinstance(act, int) else act
    args.beta = int(beta) if not isinstance(beta, bool) else (1 if beta else 0)
    args.ksplit = ksplit
    if bias is not None:
        assert bias.dtype == torch.float32
        args.bias = bias.data_ptr()
    args.bias_batch = bias_batch
    if row_map is not None:
        assert row_map.dtype == torch.int32
        args.row_map = row_map.data_ptr()
    args.bn = bn
    args.max_ctas = max_ctas
    if dynamic:
        args.tile_counter = tile_counter(C.device).data_ptr()
    _lib.check(_lib.gemm(ctypes.byref(args), _stream()), "dvgr_gemm")
    return C


# zeroed int32 counters for dynamically scheduled GEMMs: slots of ONE arena per device that the engine zeroes once per step
# (begin_step_counters); outside an engine step every call gets a fresh zeroed word
_COUNTERS = {}


def begin_step_counters(device, n=32):
    """Zeroes the per-step arena of tile counters (one fill launch) and rewinds it. Called at the start of an engine step."""
    ent = _COUNTERS.get(str(device))
    if ent is None or ent[0].numel() < n:
        ent = [torch.zeros(n, dtype=torch.int32, device=device), 0, True]
        _COUNTERS[str(device)] = ent
    else:
        ent[0].zero_()
    ent[1], ent[2] = 0, True
    return ent[0]


def end_step_counters(device):
    ent = _COUNTERS.get(str(device))
    if ent is not None:
        ent[2] = False


def tile_counter(device):
    ent = _COUNTERS.get(str(device))
    if ent is not None and ent[2] and ent[1] < ent[0].numel():
        ent[1] += 1
        return ent[0][ent[1] - 1:ent[1]]
    return torch.zeros(1, dtype=torch.int32, device=device)


def linear_fwd(x, w, bias=None, act=None, out=None, out_dtype=torch.bfloat16, bn=0):
    """y[M,N] = act(x[M,K] @ w[N,K]^T + bias). x, w bf16; bias fp32."""
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x.device)
    return gemm(x, 0, w, 0, M, N, K, out, bias=bias, act=act, bn=bn)


def linear_dgrad(dy, w, out=None, beta=False, bn=0):
    """dx[M,K] = dy[M,N] @ w[N,K]  (w read MN-major: no transposed copy)."""
    M, N = dy.shape
    K = w.shape[1]
    if out is None:
        out = torch.empty((M, K), dtype=torch.bfloat16, device=dy.device)
    return gemm(dy, 0, w, 1, M, K, N, out, beta=beta, bn=bn)


NUM_SMS = 148


def wgrad_split(rows, cols, red, batch=1):
    """(bn, ksplit) for a weight-gradient GEMM [rows, cols] reduced over `red`. The persistent kernel deals tiles
    round-robin to the 148 CTAs, so its time is ~ ceil(tiles * ksplit / 148) * (k_blocks / ksplit): pick the split that
    minimises it (smallest on ties: every split adds one atomic pass over the output)."""
    bn = 256 if (rows // 128) * ((cols + 255) // 256) * batch >= NUM_SMS else 128
    tiles = ((rows + 127) // 128) * ((cols + bn - 1) // bn) * batch
    kb = (red + 63) // 64
    best, best_cost = 1, None
    for ks in range(1, max(1, min(kb // 4, 32)) + 1):
        per = (kb + ks - 1) // ks
        cost = ((tiles * ks + NUM_SMS - 1) // NUM_SMS) * (per + 3)       # +3: pipeline fill / epilogue per tile
        if best_cost is None or cost < best_cost * 0.97:
            best, best_cost = ks, cost
    return bn, best


def linear_wgrad(dy, x, out=None, beta=False, row_map=None, bn=0, rows=None, cols=None, atomic=False, dynamic=False,
                 max_ctas=0):
    """dw[N,K] (fp32) (+)= dy[M,N]^T @ x[M,K]  (both read MN-major). atomic=True: split-K with fp32 atomic adds into
    `out` (which must already hold the value to accumulate onto, e.g. a zeroed gradient buffer)."""
    M, N = dy.shape
    K = x.shape[1]
    rows, cols = rows or N, cols or K
    if out is None:
        assert not atomic
        out = torch.empty((rows, cols), dtype=torch.float32, device=dy.device)
    if atomic:
        if DEFER_WGRAD[0] and row_map is None and not bn:
            wgrad_enqueue(dy, x, out, rows, cols)
            return out
        bn2, ks = wgrad_split(rows, cols, M)
        return gemm(dy, 1, x, 1, rows, cols, M, out, beta=2, row_map=row_map, bn=bn or bn2, ksplit=ks, dynamic=dynamic,
                    max_ctas=max_ctas)
    return gemm(dy, 1, x, 1, rows, cols, M, out, beta=beta, row_map=row_map, bn=bn, dynamic=dynamic, max_ctas=max_ctas)


# ---- deferred, grouped weight gradients. Inside a train step nothing consumes a weight gradient before the optimizer, so
#      the engine lets the autograd layer QUEUE them (DEFER_WGRAD) and flushes the queue as one persistent launch
#      (dvgr_wgrad_grouped) after backward. Outside the engine the queue is never used: linear_wgrad launches at once.
DEFER_WGRAD = [False]
_WGRAD_QUEUE = []


def wgrad_enqueue(dy, x, out, rows=None, cols=None):
    """out[rows, cols] (fp32, += ) dy[M, N]^T @ x[M, K]; the operands are kept alive until flush_wgrads()."""
    assert dy.dtype == BF16 and x.dtype == BF16 and out.dtype == F32 and dy.stride(1) == 1 and x.stride(1) == 1
    assert dy.shape[0] == x.shape[0] and out.stride(-1) == 1
    _WGRAD_QUEUE.append((dy, x, out, rows or dy.shape[1], cols or x.shape[1]))


_COLSUM_QUEUE = []


def colsum_enqueue(x, out, perm_H=0, out2=None):
    """out[C] (fp32) += column sums of x[R, C] (bf16 / fp32, last dim contiguous); x is kept alive until flush_wgrads().
    perm_H > 0: column 4j+g lands at out[g*perm_H + j] (LSTM gate de-interleave); out2: second target for the same sums."""
    assert x.dim() == 2 and x.stride(1) == 1 and out.dtype == F32 and out.is_contiguous() and out.numel() == x.shape[1]
    assert out2 is None or (out2.dtype == F32 and out2.is_contiguous() and out2.numel() == out.numel())
    _COLSUM_QUEUE.append((x, out, perm_H, out2))


_SMALL_QUEUE = []


def small_grad_enqueue(target, grad):
    """target (a bound fp32 .grad view) += grad at flush time: the gradients of the tiny parameters (attention vectors, LSTM /
    BatchNorm biases ...) accumulate in ONE scatter launch per step instead of one elementwise launch per parameter."""
    assert target.dtype == F32 and grad.dtype == F32 and target.numel() == grad.numel() and target.is_contiguous()
    _SMALL_QUEUE.append((target, grad))


def clear_deferred():
    """Drops queued (unlaunched) weight / bias gradients — called when a step aborts between enqueue and flush."""
    _WGRAD_QUEUE.clear()
    _COLSUM_QUEUE.clear()
    _SMALL_QUEUE.clear()


def flush_wgrads(keep_alive=None):
    """Launches every queued weight gradient (one grouped GEMM per 32 problems) and bias gradient (one grouped column sum).
    keep_alive: a list that receives the queued operands — for a flush on a SIDE stream, whose kernels may still be reading
    them when the caller's stream would otherwise free (and re-use) their memory."""
    if keep_alive is not None:
        keep_alive.extend([list(_SMALL_QUEUE), list(_COLSUM_QUEUE), list(_WGRAD_QUEUE)])
    if _SMALL_QUEUE:
        scatter(list(_SMALL_QUEUE), True)
        _SMALL_QUEUE.clear()
    if _COLSUM_QUEUE:
        m = len(_COLSUM_QUEUE)
        carr = (_lib.ColsumProblem * m)()
        for i, (x, out, perm_H, out2) in enumerate(_COLSUM_QUEUE):
            carr[i].in_, carr[i].in_is_f32, carr[i].ld = x.data_ptr(), 1 if x.dtype == F32 else 0, x.stride(0)
            carr[i].R, carr[i].C, carr[i].out = x.shape[0], x.shape[1], out.data_ptr()
            carr[i].perm_H, carr[i].out2 = perm_H, (out2.data_ptr() if out2 is not None else None)
        _lib.check(_lib.colsum_grouped(carr, m, _stream()), "dvgr_colsum_grouped")
        _COLSUM_QUEUE.clear()
    if not _WGRAD_QUEUE:
        return 0
    n = len(_WGRAD_QUEUE)
    arr = (_lib.WgradProblem * n)()
    for i, (dy, x, out, rows, cols) in enumerate(_WGRAD_QUEUE):
        arr[i].dy, arr[i].ld_dy, arr[i].x, arr[i].ld_x = dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0)
        arr[i].M, arr[i].rows, arr[i].cols = dy.shape[0], rows, cols
        arr[i].out, arr[i].ldc = out.data_ptr(), out.stride(-2)
    _lib.check(_lib.wgrad_grouped(arr, n, _stream()), "dvgr_wgrad_grouped")
    _WGRAD_QUEUE.clear()
    return n


def gemm_reference(A, a_rs, a_ks, B, b_rs, b_ks, M, N, K):
    C = torch.empty((M, N), dtype=torch.float32, device=A.device)
    _lib.check(_lib.gemm_reference(_ptr(A), a_rs, a_ks, _ptr(B), b_rs, b_ks, _ptr(C), N, M, N, K, _stream()),
               "dvgr_gemm_reference")
    return C


# ----------------------------------------------------------------------------------------------------- fused LSTM
def _lstm_args(gates, whh, h_hist, c_hist, S, H, T, ndir):
    a = _lib.LstmArgs()
    a.S, a.H, a.T, a.ndir = S, H, T, ndir
    a.gates, a.whh, a.h_hist, a.c_hist = gates.data_ptr(), whh.data_ptr(), h_hist.data_ptr(), c_hist.data_ptr()
    return a


def lstm_fwd(gates, whh, seq_len=None, want_seq=False):
    """Runs the T recurrent steps of all directions.
    gates [T,S,D*4H] bf16 (x W_ih^T + b, gate-interleaved; overwritten with the activated gates), whh [D,4H,H] bf16.
    Returns (h_hist [D,T+1,S,H] bf16, c_hist [D,T+1,S,H] f32, h_last [S,D*H] bf16, seq_out [S,T,D*H] bf16 | None)."""
    _check_cuda(gates, whh)
    T, S, G = gates.shape
    D, H4, H = whh.shape
    assert G == D * H4 and H4 == 4 * H and gates.is_contiguous() and whh.is_contiguous()
    dev = gates.device
    h_hist = torch.empty((D, T + 1, S, H), dtype=torch.bfloat16, device=dev)
    c_hist = torch.empty((D, T + 1, S, H), dtype=torch.float32, device=dev)
    h_hist[:, 0].zero_()
    c_hist[:, 0].zero_()
    h_last = torch.empty((S, D * H), dtype=torch.bfloat16, device=dev)
    seq_out = torch.empty((S, T, D * H), dtype=torch.bfloat16, device=dev) if want_seq else None
    a = _lstm_args(gates, whh, h_hist, c_hist, S, H, T, D)
    a.h_last, a.h_last_ld = h_last.data_ptr(), D * H
    if seq_len is not None:
        assert seq_len.dtype == torch.int32
        a.seq_len = seq_len.data_ptr()
    if seq_out is not None:
        a.seq_out, a.seq_out_ld = seq_out.data_ptr(), D * H
    st = _stream()
    for s in range(T):
        a.s = s
        _lib.check(_lib.lstm_step_fwd(ctypes.byref(a), st), "dvgr_lstm_step_fwd")
    return h_hist, c_hist, h_last, seq_out


# ---- blocked layout of the whole-sequence LSTM kernels (include/dualvgr_b200.h: dvgr_lstm_seq_fwd). The helpers below are
#      pure re-layouts (views / permutes) used by the tests and debugging tools; the train step never calls them.
def lstm_unblock_gates(gates_blk, S):
    """[T, D, RB, H/8, 4, 32, 8] bf16 -> [T, S, D*4H] (gate-interleaved columns 4*j + {i,f,g,o})."""
    T, D, RB, UG = gates_blk.shape[:4]
    return gates_blk.permute(0, 2, 5, 1, 3, 4, 6).reshape(T, RB * 32, D * UG * 32)[:, :S]


def lstm_block_gates(gates, D):
    """[T, S, D*4H] -> blocked [T, D, RB, H/8, 4, 32, 8] (rows padded to a multiple of 32 with zeros)."""
    T, S, G = gates.shape
    RB, UG = (S + 31) // 32, G // D // 32
    g = torch.zeros((T, RB * 32, G), dtype=gates.dtype, device=gates.device)
    g[:, :S] = gates
    return g.view(T, RB, 32, D, UG, 4, 8).permute(0, 3, 1, 4, 5, 2, 6).contiguous()


def lstm_unblock_c(c_blk, S):
    """[D, T+1, RB, H/8, 2, 32, 4] f32 -> [D, T+1, S, H]."""
    D, T1, RB, UG = c_blk.shape[:4]
    return c_blk.permute(0, 1, 2, 5, 3, 4, 6).reshape(D, T1, RB * 32, UG * 8)[:, :, :S]


def lstm_block_c(c, ):
    """[D, T+1, S, H] -> blocked [D, T+1, RB, H/8, 2, 32, 4]."""
    D, T1, S, H = c.shape
    RB, UG = (S + 31) // 32, H // 8
    x = torch.zeros((D, T1, RB * 32, H), dtype=c.dtype, device=c.device)
    x[:, :, :S] = c
    return x.view(D, T1, RB, 32, UG, 2, 4).permute(0, 1, 2, 4, 5, 3, 6).contiguous()


# SMs left free by the persistent launch of the appearance encoder's backward recurrence for the kernels that run next to it
# on other streams: the question encoder's backward and, with more than one rank, the NCCL all-reduce of the early gradient
# bucket. The engine sets it (32); 0 = take every SM.
RESERVE_SMS = [0]


def _cap(which=0):
    """Grid cap of the appearance encoder's backward launches: which = 0 the recurrence, 1 the weight-gradient GEMMs (only
    capped when DVGR_RESERVE_WGRAD=1: they start when the question encoder's recurrence is nearly done)."""
    if which == 1 and os.environ.get("DVGR_RESERVE_WGRAD", "0") == "0":
        return 0
    return NUM_SMS - RESERVE_SMS[0] if RESERVE_SMS[0] > 0 else 0


def lstm_seq_fwd(x, wih, whh, bias, K1=None, seq_len=None, want_seq=False, h_last=None):
    """Whole-sequence fused forward (ONE persistent launch): x [T,S,ld] bf16 time-major, wih [D*4H, ld'] bf16 and
    whh [D,4H,H] bf16 gate-interleaved, bias [D*4H] f32 (b_ih + b_hh, interleaved).
    Returns (gates_blk ACTIVATED [T,D,RB,H/8,4,32,8] bf16, h_hist [D,T+1,S,H] bf16, c_blk [D,T+1,RB,H/8,2,32,4] f32,
    h_last [S,D*H], seq_out | None, sync); gates_blk / c_blk are in the kernels' blocked layout (lstm_unblock_*);
    sync[-1] is the kernel's sticky dependency-timeout flag (0 in a healthy run)."""
    _check_cuda(x, wih, whh, bias)
    T, S, ldx = x.shape
    D, H4, H = whh.shape
    K1 = K1 or ldx
    assert x.dtype == BF16 and wih.dtype == BF16 and whh.dtype == BF16 and bias.dtype == F32
    assert x.is_contiguous() and wih.stride(1) == 1 and whh.is_contiguous() and wih.shape[0] == D * H4 and H4 == 4 * H
    dev = x.device
    RB, UG = (S + 31) // 32, H // 8
    gates = torch.empty((T, D, RB, UG, 4, 32, 8), dtype=BF16, device=dev)
    # slot 0 (the initial state) of h_hist / c_hist is implicit zeros: the whole-sequence kernels never read it, and the W_hh
    # weight gradient skips it (its contribution is zero) — no fill launches
    h_hist = torch.empty((D, T + 1, S, H), dtype=BF16, device=dev)
    c_hist = torch.empty((D, T + 1, RB, UG, 2, 32, 4), dtype=F32, device=dev)
    if h_last is None:
        h_last = torch.empty((S, D * H), dtype=BF16, device=dev)
    assert h_last.dtype == BF16 and tuple(h_last.shape) == (S, D * H) and h_last.is_contiguous()
    seq_out = torch.empty((S, T, D * H), dtype=BF16, device=dev) if want_seq else None
    sync = torch.zeros((int(_lib.lib.dvgr_lstm_seq_sync_words(S, D)),), dtype=torch.int32, device=dev)
    a = _lib.LstmSeqArgs()
    l = a.lstm
    l.S, l.H, l.T, l.ndir, l.s = S, H, T, D, 0
    l.gates, l.whh, l.h_hist, l.c_hist = gates.data_ptr(), whh.data_ptr(), h_hist.data_ptr(), c_hist.data_ptr()
    l.h_last, l.h_last_ld = h_last.data_ptr(), D * H
    if seq_len is not None:
        assert seq_len.dtype == torch.int32
        l.seq_len = seq_len.data_ptr()
    if seq_out is not None:
        l.seq_out, l.seq_out_ld = seq_out.data_ptr(), D * H
    a.x, a.x_ld, a.K1 = x.data_ptr(), ldx, K1
    a.wih, a.wih_ld = wih.data_ptr(), wih.stride(0)
    a.bias, a.sync = bias.data_ptr(), sync.data_ptr()
    _lib.check(_lib.lstm_seq_fwd(ctypes.byref(a), _stream()), "dvgr_lstm_seq_fwd")
    return gates, h_hist, c_hist, h_last, seq_out, sync


def lstm_bwd(gates, whh, h_hist, c_hist, dh_last, seq_len=None, dh_seq=None, whole_sequence=False, dh_seq_blocked=None,
             max_ctas=0):
    """Backward through the T steps.
    per-step path: `gates` [T,S,D*4H] (activated gates from lstm_fwd) is overwritten in place with the pre-activation gate
    gradients, which feed the W_ih / W_hh / bias wgrads; returns gates.
    whole_sequence: one persistent launch for steps T-2..0 (dvgr_lstm_seq_bwd); `gates` / `c_hist` are the BLOCKED tensors of
    lstm_seq_fwd; returns (dgates [T,S,D*4H] bf16, sync) with sync[-1] the sticky dependency-timeout flag."""
    _check_cuda(gates, whh, dh_last)
    D, H4, H = whh.shape
    if whole_sequence:
        T, S = gates.shape[0], h_hist.shape[2]
        RB, UG = (S + 31) // 32, H // 8
        assert tuple(gates.shape) == (T, D, RB, UG, 4, 32, 8) and tuple(c_hist.shape) == (D, T + 1, RB, UG, 2, 32, 4)
        # ONE zero-filled arena for everything that must start at zero (running dc, dh carry, sync words): one fill launch
        n_run = D * RB * UG * 256
        n_sync = int(_lib.lib.dvgr_lstm_seq_sync_words(S, D))
        arena = torch.zeros((2 * n_run + n_sync + 3,), dtype=torch.float32, device=gates.device)
        dc = arena[:n_run].view(D, RB, UG, 2, 32, 4)
    else:
        T, S, G = gates.shape
        dc = torch.zeros((D, S, H), dtype=torch.float32, device=gates.device)
    a = _lstm_args(gates, whh, h_hist, c_hist, S, H, T, D)
    a.max_ctas = max_ctas
    a.dc = dc.data_ptr()
    if dh_last is not None:
        assert dh_last.dtype == torch.bfloat16 and dh_last.stride(-1) == 1
        a.dh_last, a.dh_last_ld = dh_last.data_ptr(), dh_last.stride(0)
    if seq_len is not None:
        a.seq_len = seq_len.data_ptr()
        carry = (arena[n_run:2 * n_run].view(D, RB, UG, 2, 32, 4) if whole_sequence
                 else torch.zeros((D, S, H), dtype=torch.float32, device=gates.device))
        a.dh_carry = carry.data_ptr()
    if dh_seq_blocked is not None:      # already in the kernels' blocked layout (lstm_pack_dh)
        assert whole_sequence and tuple(dh_seq_blocked.shape) == (T, D, RB, UG, 32, 8) and dh_seq_blocked.is_contiguous()
        a.dh_seq, a.seq_out_ld = dh_seq_blocked.data_ptr(), D * H
    elif dh_seq is not None:
        if whole_sequence:      # [S, T, D*H] -> blocked [T, D, RB, H/8, 32, 8]: one 512-byte warp access per (row block, unit group)
            assert tuple(dh_seq.shape) == (S, T, D * H) and dh_seq.dtype == BF16
            pad = torch.zeros((RB * 32, T, D * H), dtype=BF16, device=gates.device)
            pad[:S] = dh_seq
            dh_seq = pad.view(RB, 32, T, D, UG, 8).permute(2, 3, 0, 4, 1, 5).contiguous()
        a.dh_seq, a.seq_out_ld = dh_seq.data_ptr(), D * H
    st = _stream()
    if whole_sequence:
        dgates = torch.empty((T, S, D * H4), dtype=BF16, device=gates.device)
        sync = arena[2 * n_run:2 * n_run + n_sync].view(torch.int32)
        _lib.check(_lib.lstm_seq_bwd(ctypes.byref(a), _ptr(dgates), _ptr(sync), st), "dvgr_lstm_seq_bwd")
        return dgates, sync
    for s in range(T - 1, -1, -1):
        a.s = s
        _lib.check(_lib.lstm_step_bwd(ctypes.byref(a), st), "dvgr_lstm_step_bwd")
    return gates


# ======================================================================================================================
# raw wrappers of the fused kernels (used directly by the per-kernel parity tests, and by the autograd layer below)
# ======================================================================================================================
def _empty(shape, dtype, like):
    return torch.empty(shape, dtype=dtype, device=like.device)


def _v(name, t):
    """Entry point `name` for the activation dtype of tensor t (bf16: the default build; fp32: the _f32 variant)."""
    dt = t if isinstance(t, torch.dtype) else t.dtype
    assert dt in (BF16, F32), dt
    return _lib.variant(name, dt == F32)


def colsum(x, out=None, accumulate=False, scale=1.0):
    """out[C] (+)= scale * sum over rows of x[R, C] (bf16 or fp32, last dim contiguous)."""
    assert x.dim() == 2 and x.stride(1) == 1
    if DEFER_WGRAD[0] and accumulate and out is not None and scale == 1.0:
        colsum_enqueue(x, out)       # a bias gradient inside an engine step: grouped with the others at flush time
        return out
    R, C = x.shape
    ws = _empty((int(_lib.lib.dvgr_colsum_workspace(R, C)),), F32, x)
    if out is None:
        out = _empty((C,), F32, x)
    _lib.check(_lib.colsum(_ptr(x), 1 if x.dtype == F32 else 0, x.stride(0), R, C, _ptr(ws), _ptr(out),
                           1 if accumulate else 0, float(scale), _stream()), "dvgr_colsum")
    return out


def colsum_batched(x):
    """out[g][C] = sum over rows of x[g][R, C] for a contiguous [G, R, C] tensor (bf16 or fp32): ONE launch pair for all g."""
    assert x.dim() == 3 and x.is_contiguous()
    G, R, C = x.shape
    ws = _empty((G * int(_lib.lib.dvgr_colsum_workspace(R, C)),), F32, x)
    out = _empty((G, C), F32, x)
    _lib.check(_lib.colsum_batched(_ptr(x), 1 if x.dtype == F32 else 0, C, R * C, R, C, G, _ptr(ws), _ptr(out), C, 0, 1.0,
                                   _stream()), "dvgr_colsum_batched")
    return out


def cast_rows(w, out=None, out_cols=None, lstm_H=0):
    """fp32 [R, C] -> bf16 [R, out_cols] (zero padded); lstm_H>0 interleaves LSTM gate rows (4j+g <- g*H+j)."""
    assert w.dtype == F32 and w.dim() == 2 and w.stride(1) == 1
    R, C = w.shape
    oc = out_cols or C
    if out is None:
        out = _empty((R, oc), BF16, w)
    assert out.stride(1) == 1
    _lib.check(_lib.cast_rows(_ptr(w), w.stride(0), _ptr(out), out.stride(0), R, C, oc, lstm_H, _stream()), "dvgr_cast_rows")
    return out


def prep_features(x, T, do_tanh, time_major, p=0.0, seed=0, stream_id=0, out_dtype=BF16):
    """x fp32 [S*T, C] (S sequences of T steps) -> bf16 [T*S, C] (time_major) / [S*T, C]: tanh(dropout(x)) in one pass."""
    assert x.dtype in (F32, BF16) and x.is_contiguous()
    C = x.shape[-1]
    rows = x.numel() // C
    S = rows // T
    out = _empty((rows, C), out_dtype, x)
    _lib.check(_v("prep_features_ex", out_dtype)(_ptr(x), 1 if x.dtype == BF16 else 0, _ptr(out), S, T, C, 1 if do_tanh else 0,
                                     1 if time_major else 0, float(p), int(seed), int(stream_id), _stream()),
               "dvgr_prep_features_ex")
    return out


def prep_features_gather(store, rows, T, do_tanh, time_major, p=0.0, seed=0, stream_id=0, err=None, out_dtype=BF16):
    """prep_features of the batch store[rows] read straight from a device-resident store: store [V, N, T, C] (or [V, N, C]
    with T = 1) fp32 / bf16, rows [B] int32 -> [B*N*T, C] laid out as prep_features lays it out. A row outside [0, V)
    reads nothing, gives zero output rows and sets err ([1] int32, sticky)."""
    _check_cuda(store, rows, err)
    assert store.dtype in (F32, BF16) and store.is_contiguous() and store.dim() in (3, 4)
    assert (store.shape[2] if store.dim() == 4 else 1) == T, (tuple(store.shape), T)
    assert rows.dtype == torch.int32 and rows.dim() == 1 and rows.is_contiguous()
    assert err is not None and err.dtype == torch.int32 and err.numel() >= 1
    V, N, C = store.shape[0], store.shape[1], store.shape[-1]
    B = rows.numel()
    out = _empty((B * N * T, C), out_dtype, store)
    _lib.check(_v("prep_features_gather", out_dtype)(_ptr(store), 1 if store.dtype == BF16 else 0, V, N, _ptr(rows), B,
                                                     _ptr(out), T, C, 1 if do_tanh else 0, 1 if time_major else 0, float(p),
                                                     int(seed), int(stream_id), _ptr(err), _stream()),
               "dvgr_prep_features_gather")
    return out


def dropout_raw(x, p, seed, stream_id, out=None):
    assert x.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    assert out.dtype == x.dtype
    _lib.check(_v("dropout", x)(_ptr(x), _ptr(out), x.numel(), float(p), int(seed), int(stream_id), _stream()), "dvgr_dropout")
    return out


def act_bwd(dy, y, act, out=None, accumulate=False, p=0.0, seed=0, stream_id=0):
    """out (+)= dy * dropout_mask * act'(y) with y the activation output."""
    assert dy.is_contiguous() and (y is None or y.dtype == dy.dtype)
    if out is None:
        out = torch.empty_like(dy)
    a = _ACT[act] if not isinstance(act, int) else act
    _lib.check(_v("act_bwd", dy)(_ptr(dy), _ptr(y) if y is not None else _ptr(dy), _ptr(out), dy.numel(), a,
                            1 if accumulate else 0, float(p), int(seed), int(stream_id), _stream()), "dvgr_act_bwd")
    return out


def scatter(pairs, accumulate):
    """pairs: list of (dst, src) fp32 tensors of equal numel, dst contiguous: dst (+)= src for all of them, 64 per launch."""
    if not pairs:
        return
    arr = (_lib.Seg * len(pairs))()
    keep = []
    for i, (d, s_) in enumerate(pairs):
        s_ = s_ if s_.is_contiguous() else s_.contiguous()
        keep.append(s_)
        assert d.dtype == F32 and s_.dtype == F32 and d.is_contiguous() and d.numel() == s_.numel() and d.is_cuda and s_.is_cuda
        arr[i].dst, arr[i].src, arr[i].n = d.data_ptr(), s_.data_ptr(), d.numel()
    _lib.check(_lib.scatter(arr, len(pairs), 1 if accumulate else 0, _stream()), "dvgr_scatter")


def scatter_add(pairs):
    scatter(pairs, True)


def add_(a, b):
    assert a.dtype == b.dtype and a.is_contiguous() and b.is_contiguous() and a.numel() == b.numel()
    _lib.check(_v("add", a)(_ptr(a), _ptr(b), a.numel(), _stream()), "dvgr_add")
    return a


def qattn_fwd(y, wf, cf, qlen, words, W, ld_qc):
    B, L, D = y.shape
    alpha, nrm, prob = (_empty((B, L), F32, y) for _ in range(3))
    ssum = _empty((B,), F32, y)
    qc = _empty((B, ld_qc), y.dtype, y)
    assert words.dtype == y.dtype
    _lib.check(_v("qattn_fwd", y)(_ptr(y), _ptr(wf), _ptr(cf), _ptr(qlen), _ptr(words), words.stride(1), B, L, D, W,
                              _ptr(alpha), _ptr(nrm), _ptr(prob), _ptr(ssum), _ptr(qc), ld_qc, _stream()), "dvgr_qattn_fwd")
    return qc, alpha, nrm, prob, ssum


def qattn_bwd(dqc, y, wf, qlen, words, W, alpha, nrm, prob, ssum, dwords=None, raw=False):
    """raw=True: returns the per-sample partials (dwf_part [B, D], dcf_part [B, 1]) instead of their column sums."""
    B, L, D = y.shape
    dy = torch.empty_like(y)
    acc = dwords is not None
    if dwords is None:
        dwords = torch.zeros_like(words)
    dwf_part = _empty((B, D), F32, y)
    dcf_part = _empty((B, 1), F32, y)
    assert dqc.dtype == y.dtype
    _lib.check(_v("qattn_bwd", y)(_ptr(dqc), dqc.stride(0), _ptr(y), _ptr(wf), _ptr(qlen), _ptr(words), words.stride(1), B, L,
                              D, W, _ptr(alpha), _ptr(nrm), _ptr(prob), _ptr(ssum), _ptr(dy), _ptr(dwords),
                              1 if acc else 0, _ptr(dwf_part), _ptr(dcf_part), _stream()), "dvgr_qattn_bwd")
    if raw:
        return dy, dwords, dwf_part, dcf_part
    return dy, dwords, colsum(dwf_part), colsum(dcf_part)


def gate_fwd(xa, xm, query):
    B, N, D = xa.shape
    ga, gm = _empty((B, N), F32, xa), _empty((B, N), F32, xa)
    assert xm.dtype == xa.dtype == query.dtype
    _lib.check(_v("gate_fwd", xa)(_ptr(xa), _ptr(xm), _ptr(query), query.stride(0), B, N, D, _ptr(ga), _ptr(gm), _stream()),
               "dvgr_gate_fwd")
    return ga, gm


def gate_bwd(xa, xm, query, ga, gm, dga, dga2, dgm, dgm2, dxa, dxm, dquery=None):
    """dxa / dxm are accumulated into; returns dquery [B, ld_q] (written into `dquery` when given: same strides as query)."""
    B, N, D = xa.shape
    if dquery is None:
        dquery = torch.empty_like(query)
    assert dquery.shape == query.shape and dquery.stride() == query.stride() and dquery.dtype == query.dtype
    assert dxa.dtype == xa.dtype and dxm.dtype == xa.dtype
    _lib.check(_v("gate_bwd", xa)(_ptr(xa), _ptr(xm), _ptr(query), query.stride(0), B, N, D, _ptr(ga), _ptr(gm), _ptr(dga),
                             _ptr(dga2), _ptr(dgm), _ptr(dgm2), _ptr(dxa), _ptr(dxm), _ptr(dquery), _stream()),
               "dvgr_gate_bwd")
    return dquery


def _gat_args(whs, gates, avecs, outs, adj, B, N, D, heads, slope, p_att, p_out, seed, streams):
    a = _lib.GatArgs()
    a.n_graphs = len(whs)
    a.B, a.N, a.D, a.heads = B, N, D, heads
    a.ld_wh, a.ld_out = whs[0].stride(-2), outs[0].stride(-2)
    a.adj = adj.data_ptr()
    a.slope, a.p_att, a.p_out, a.seed = slope, p_att, p_out, seed
    for i in range(len(whs)):
        g = a.graphs[i]
        g.wh, g.gate, g.avec, g.out = whs[i].data_ptr(), gates[i].data_ptr(), avecs[i].data_ptr(), outs[i].data_ptr()
        g.drop_stream = streams[i]
    return a


def gat_attn_fwd(whs, gates, avecs, adj, B, N, heads=4, slope=0.01, p_att=0.0, p_out=0.0, seed=0, streams=None,
                 outs=None, want_f32=False):
    """whs: list of [B*N, D] bf16 (row stride free), gates: list of [B, N] f32, avecs: list of [heads, 2*Dh+1] f32."""
    D = whs[0].shape[-1]
    G = len(whs)
    streams = streams or [2 * i for i in range(G)]
    if outs is None:
        outs = [_empty((B * N, D), whs[0].dtype, whs[0]) for _ in range(G)]
    a = _gat_args(whs, gates, avecs, outs, adj, B, N, D, heads, slope, p_att, p_out, seed, streams)
    outs32 = None
    if want_f32:
        outs32 = [_empty((B, N, D), F32, whs[0]) for _ in range(G)]
        for i in range(G):
            a.graphs[i].out_f32 = outs32[i].data_ptr()
    _lib.check(_v("gat_attn_fwd", whs[0])(ctypes.byref(a), _stream()), "dvgr_gat_attn_fwd")
    return outs, outs32


def gat_attn_bwd(whs, gates, avecs, outs, douts, adj, B, N, heads=4, slope=0.01, p_att=0.0, p_out=0.0, seed=0,
                 streams=None, douts32=None, dwhs=None, raw=False):
    D = whs[0].shape[-1]
    G = len(whs)
    Dh = D // heads
    streams = streams or [2 * i for i in range(G)]
    a = _gat_args(whs, gates, avecs, outs, adj, B, N, D, heads, slope, p_att, p_out, seed, streams)
    if dwhs is None:
        dwhs = [torch.empty_like(w) for w in whs]
    dgates = [_empty((B, N), F32, whs[0]) for _ in range(G)]
    dav_all = _empty((G, B, heads * (2 * Dh + 1)), F32, whs[0])
    dav_part = [dav_all[i] for i in range(G)]
    for i in range(G):
        g = a.graphs[i]
        assert dwhs[i].stride(-2) == whs[i].stride(-2) and douts[i].stride(-2) == outs[i].stride(-2)
        g.dout, g.dwh, g.dgate, g.davec = douts[i].data_ptr(), dwhs[i].data_ptr(), dgates[i].data_ptr(), dav_part[i].data_ptr()
        if douts32 is not None and douts32[i] is not None:
            g.dout_f32 = douts32[i].data_ptr()
    _lib.check(_v("gat_attn_bwd", whs[0])(ctypes.byref(a), _stream()), "dvgr_gat_attn_bwd")
    if raw:                                             # per-video partials [G, B, heads * (2 Dh + 1)]: the caller reduces them
        return dwhs, dgates, dav_all
    dav = colsum_batched(dav_all)                       # per-video partial sums -> [G, heads * (2 Dh + 1)] in one launch pair
    davecs = [dav[i].view(heads, 2 * Dh + 1) for i in range(G)]
    return dwhs, dgates, davecs


def view_attn_fwd(hidden, z, x, w2, want_embed=True):
    """hidden, z: [2, M, D] bf16; x [M, D] bf16; w2 [D] f32."""
    _, M, D = z.shape
    xnew = torch.empty_like(x)
    embed = torch.empty_like(x) if want_embed else None
    beta = _empty((M, 2), F32, x)
    _lib.check(_v("view_attn_fwd", z)(_ptr(hidden), _ptr(z), _ptr(x), _ptr(w2), M, D, _ptr(xnew), _ptr(embed), _ptr(beta),
                                  _stream()), "dvgr_view_attn_fwd")
    return xnew, embed, beta


def view_attn_bwd(dxnew, dembed, hidden, z, w2, beta):
    _, M, D = z.shape
    dz, dhid = torch.empty_like(z), torch.empty_like(hidden)
    blocks = int(_lib.lib.dvgr_view_attn_bwd_blocks(M))
    part = _empty((blocks, D), F32, z)
    _lib.check(_v("view_attn_bwd", z)(_ptr(dxnew), _ptr(dembed), _ptr(hidden), _ptr(z), _ptr(w2), _ptr(beta), M, D, _ptr(dz),
                                  _ptr(dhid), _ptr(part), _stream()), "dvgr_view_attn_bwd")
    return dz, dhid, colsum(part)


def mfb_fwd(x0, x1):
    M, mm2 = x0.shape
    z = _empty((M, mm2 // 2), x0.dtype, x0)
    _lib.check(_v("mfb_fwd", x0)(_ptr(x0), _ptr(x1), _ptr(z), M, mm2, _stream()), "dvgr_mfb_fwd")
    return z


def mfb_bwd(dz, x0, x1):
    M, mm2 = x0.shape
    d0, d1 = torch.empty_like(x0), torch.empty_like(x1)
    _lib.check(_v("mfb_bwd", x0)(_ptr(dz), _ptr(x0), _ptr(x1), _ptr(d0), _ptr(d1), M, mm2, _stream()), "dvgr_mfb_bwd")
    return d0, d1


def readout_fwd(v, u, w, c, pooled=None):
    B, N, D = v.shape
    alpha = _empty((B, N), F32, v)
    if pooled is None:
        pooled = _empty((B, D), v.dtype, v)
    _lib.check(_v("readout_fwd", v)(_ptr(v), _ptr(u), _ptr(w), _ptr(c), B, N, D, _ptr(alpha), _ptr(pooled), pooled.stride(0),
                                _stream()), "dvgr_readout_fwd")
    return pooled, alpha


def readout_bwd(dpooled, v, u, w, alpha, raw=False):
    """raw=True: returns the per-sample partials (dw_part [B, D], dc_part [B, 1]) instead of their column sums."""
    B, N, D = v.shape
    dv, du = torch.empty_like(v), torch.empty_like(u)
    dw_part, dc_part = _empty((B, D), F32, v), _empty((B, 1), F32, v)
    _lib.check(_v("readout_bwd", v)(_ptr(dpooled), dpooled.stride(0), _ptr(v), _ptr(u), _ptr(w), _ptr(alpha), B, N, D, _ptr(dv),
                                _ptr(du), _ptr(dw_part), _ptr(dc_part), _stream()), "dvgr_readout_bwd")
    if raw:
        return dv, du, dw_part, dc_part
    return dv, du, colsum(dw_part), colsum(dc_part)


def bn_stats(x):
    """[2, D] f32: per-column (sum, sum of squares) of x [B, D] — the operand of the SyncBN all-reduce."""
    B, D = x.shape
    out = _empty((2, D), F32, x)
    _lib.check(_lib.bn_stats(_ptr(x), 1 if x.dtype == F32 else 0, B, D, _ptr(out), _stream()), "dvgr_bn_stats")
    return out


def bn_fwd(x, gamma, beta, run_mean, run_var, training, momentum=0.1, eps=1e-5, ext_stats=None, Btot=0, out_dtype=BF16):
    """ext_stats [2, D] = all-reduced bn_stats over a global batch of Btot rows (synchronised BatchNorm)."""
    B, D = x.shape
    y = _empty((B, D), out_dtype, x)
    mean, rstd = _empty((D,), F32, x), _empty((D,), F32, x)
    _lib.check(_v("bn_fwd_ex", out_dtype)(_ptr(x), 1 if x.dtype == F32 else 0, B, D, _ptr(gamma), _ptr(beta), _ptr(run_mean), _ptr(run_var),
                              1 if training else 0, momentum, eps, _ptr(y), _ptr(mean), _ptr(rstd), _ptr(ext_stats),
                              Btot if ext_stats is not None else B, _stream()), "dvgr_bn_fwd")
    return y, mean, rstd


def bn_bwd(dy, x, gamma, mean, rstd, training, ext_sums=None, Btot=0, stats_only=False):
    """stats_only: returns (None, local sum dy*xhat, local sum dy) without dx; ext_sums [2, D] = (sum dy, sum dy*xhat) over the
    global batch of Btot rows: dx of the synchronised BatchNorm."""
    B, D = x.shape
    dx = None if stats_only else torch.empty_like(x)
    dgamma, dbeta = _empty((D,), F32, x), _empty((D,), F32, x)
    assert dy.dtype == BF16 or x.dtype == F32
    _lib.check(_v("bn_bwd_ex", dy)(_ptr(dy), _ptr(x), 1 if x.dtype == F32 else 0, B, D, _ptr(gamma), _ptr(mean), _ptr(rstd),
                              1 if training else 0, _ptr(dx), _ptr(dgamma), _ptr(dbeta), _ptr(ext_sums),
                              Btot if ext_sums is not None else B, 1 if stats_only else 0, _stream()), "dvgr_bn_bwd")
    return dx, dgamma, dbeta


def cross_entropy(logits, answers, scale=1.0, want_grad=True, grad_f32=False):
    """Mean CE over the batch. Returns (loss scalar tensor, dlogits, correct [B] int32); dlogits is [B, A8] bf16 (A padded to
    8: a GEMM operand) or, with grad_f32, [B, A] fp32 (the gradient of the fp32 logits as autograd passes it on)."""
    B, A = logits.shape
    assert logits.dtype == F32 and logits.is_contiguous() and answers.dtype == torch.int64
    A8 = A if grad_f32 else (A + 7) // 8 * 8
    part = _empty((B, 1), F32, logits)
    dlog = _empty((B, A8), F32 if grad_f32 else BF16, logits) if want_grad else None
    correct = torch.empty((B,), dtype=torch.int32, device=logits.device)
    _lib.check(_lib.cross_entropy_ex(_ptr(logits), _ptr(answers), B, A, float(scale), _ptr(part), _ptr(dlog),
                                     1 if grad_f32 else 0, A8, _ptr(correct), _stream()), "dvgr_cross_entropy")
    return colsum(part)[0], dlog, correct


def pair_loss_multi(jobs, B, N, D, like):
    """jobs: list of dicts(x, y, mode, coef, dx, dy, acc_x, acc_y). Returns per-job loss sums as a [n_jobs] f32 tensor."""
    n = len(jobs)
    arr = (_lib.PairJob * n)()
    part = _empty((B, n), F32, like)
    for i, j in enumerate(jobs):
        assert j["x"].dtype == F32 and j["y"].dtype == F32 and j["x"].is_contiguous() and j["y"].is_contiguous()
        arr[i].x, arr[i].y = j["x"].data_ptr(), j["y"].data_ptr()
        arr[i].dx = j["dx"].data_ptr() if j.get("dx") is not None else None
        arr[i].dy = j["dy"].data_ptr() if j.get("dy") is not None else None
        arr[i].loss_part, arr[i].loss_col, arr[i].loss_ld = part.data_ptr(), i, n
        arr[i].mode, arr[i].coef = j["mode"], float(j["coef"])
        arr[i].accumulate_x, arr[i].accumulate_y = j.get("acc_x", 0), j.get("acc_y", 0)
    ws = _empty((int(_lib.lib.dvgr_pair_loss_workspace(n, B, N, D)),), F32, like)
    _lib.check(_lib.pair_loss_multi(arr, n, B, N, D, _ptr(ws), _stream()), "dvgr_pair_loss_multi")
    return colsum(part)


def aux_loss_unit(ca, cm, aq, mq, coef_com, coef_dep, want_grad=True, precise=False):
    """The three auxiliary terms of one DualVGR unit (tensor-centric kernels). Inputs fp32 [B, N, D] contiguous.
    Returns (vals [3] f32 = coef-scaled (common, HSIC(aq, ca), HSIC(mq, cm)), (d_ca, d_cm, d_aq, d_mq) | None)."""
    B, N, D = ca.shape
    for t in (ca, cm, aq, mq):
        assert t.dtype == F32 and t.is_contiguous() and tuple(t.shape) == (B, N, D)
    grads = tuple(torch.empty_like(t) for t in (ca, cm, aq, mq)) if want_grad else (None,) * 4
    part = _empty((B, 3), F32, ca)
    ws = _empty((int(_lib.lib.dvgr_aux_loss_workspace(B, N, D)),), F32, ca)
    _lib.check(_lib.aux_loss_unit_ex(_ptr(ca), _ptr(cm), _ptr(aq), _ptr(mq), float(coef_com), float(coef_dep), B, N, D,
                                     _ptr(grads[0]), _ptr(grads[1]), _ptr(grads[2]), _ptr(grads[3]), _ptr(part), _ptr(ws),
                                     1 if precise else 0, _stream()), "dvgr_aux_loss_unit_ex")
    return colsum(part), (grads if want_grad else None)


def aux_loss_workspace(B, N, D, like):
    return _empty((int(_lib.lib.dvgr_aux_loss_workspace(B, N, D)),), F32, like)


def aux_loss_unit_into(ca, cm, aq, mq, coef_com, coef_dep, g_ca, g_cm, g_aq, g_mq, part, ws):
    """aux_loss_unit with caller-owned outputs: gradients g_* (like the inputs), per-sample partial values part [B, 3]
    (column sums = the three coef-scaled terms), workspace ws (aux_loss_workspace). Launches on the CURRENT stream, which may
    be a side stream: nothing is allocated here."""
    B, N, D = ca.shape
    for t in (ca, cm, aq, mq, g_ca, g_cm, g_aq, g_mq):
        assert t.dtype == F32 and t.is_contiguous() and tuple(t.shape) == (B, N, D)
    assert part.dtype == F32 and part.is_contiguous() and part.numel() == 3 * B
    _lib.check(_lib.aux_loss_unit(_ptr(ca), _ptr(cm), _ptr(aq), _ptr(mq), float(coef_com), float(coef_dep), B, N, D,
                                  _ptr(g_ca), _ptr(g_cm), _ptr(g_aq), _ptr(g_mq), _ptr(part), _ptr(ws), _stream()),
               "dvgr_aux_loss_unit")


def pair_loss(x, y, mode, coef, dx=None, dy=None, want_grad=True):
    """mode 0: coef * sum (G_x - G_y)^2 ; mode 1: coef * HSIC. x, y fp32 [B, N, D]. dx / dy given => accumulated into.
    Returns (loss scalar tensor, dx, dy)."""
    B, N, D = x.shape
    accx, accy = dx is not None, dy is not None
    if want_grad:
        dx = dx if accx else torch.empty_like(x)
        dy = dy if accy else torch.empty_like(y)
    job = dict(x=x, y=y, mode=mode, coef=coef, dx=dx if want_grad else None, dy=dy if want_grad else None,
               acc_x=1 if accx else 0, acc_y=1 if accy else 0)
    return pair_loss_multi([job], B, N, D, x)[0], dx, dy


def sumsq(g):
    ws = _empty((int(_lib.lib.dvgr_sumsq_blocks()),), F32, g)
    out = _empty((1,), F32, g)
    _lib.check(_lib.sumsq(_ptr(g), g.numel(), _ptr(ws), _ptr(out), _stream()), "dvgr_sumsq")
    return out


def adam_step(p, g, m, v, lr, step, beta1=0.9, beta2=0.999, eps=1e-8, max_norm=0.0, norm_sq=None, grad_scale=1.0,
              step_dev=None, shadow=None):
    _lib.check(_lib.adam_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), lr, beta1, beta2, eps, step, max_norm,
                              _ptr(norm_sq), grad_scale, _ptr(step_dev), _ptr(shadow), _stream()), "dvgr_adam_step")


# ---------------------------------------------------------------------------------------- multi-stream / packing helpers
def _parr(ts):
    arr = (ctypes.c_void_p * len(ts))()
    for i, t in enumerate(ts):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


def _uarr(vals):
    arr = (ctypes.c_uint * len(vals))()
    for i, v in enumerate(vals):
        arr[i] = int(v)
    return arr


def dropout_multi(ins, outs, streams, p, seed):
    """outs[i] = ins[i] * mask(seed, streams[i]) for up to 4 bf16 tensors of equal size in ONE launch."""
    n = ins[0].numel()
    for a, b in zip(ins, outs):
        assert a.dtype == BF16 and b.dtype == BF16 and a.is_contiguous() and b.is_contiguous() and a.numel() == n == b.numel()
    _lib.check(_lib.dropout_multi(_parr(ins), _parr(outs), _uarr(streams), len(ins), n, float(p), int(seed), _stream()),
               "dvgr_dropout_multi")
    return outs


def gat_input_bwd(dxts, streams, per_stream, bases, outs, p, seed):
    """outs[s] = bases[s] + sum_j mask(streams[s*per_stream+j]) * dxts[s*per_stream+j] (bf16, one launch for all streams)."""
    n = outs[0].numel()
    for t in list(dxts) + list(outs) + [b for b in bases if b is not None]:
        assert t.dtype == BF16 and t.is_contiguous() and t.numel() == n
    _lib.check(_lib.gat_input_bwd(_parr(dxts), _uarr(streams), len(outs), per_stream, _parr(bases), _parr(outs), n, float(p),
                                  int(seed), _stream()), "dvgr_gat_input_bwd")
    return outs


def embed_fwd(tokens, table, Wp, p=0.0, seed=0, stream_id=0, out_dtype=BF16):
    """words [B, L, Wp] bf16 and time-major x [L, B, Wp] bf16 = tanh(dropout(table[tokens])), zero-padded to Wp columns."""
    _check_cuda(tokens, table)
    B, L = tokens.shape
    V, W = table.shape
    assert tokens.dtype == torch.int64 and tokens.is_contiguous() and table.dtype == F32 and table.is_contiguous()
    words = torch.empty((B, L, Wp), dtype=out_dtype, device=table.device)
    x_tm = torch.empty((L, B, Wp), dtype=out_dtype, device=table.device)
    _lib.check(_v("embed_fwd", out_dtype)(_ptr(tokens), _ptr(table), B, L, W, Wp, _ptr(words), _ptr(x_tm), float(p), int(seed),
                              int(stream_id), _stream()), "dvgr_embed_fwd")
    return words, x_tm


def embed_bwd(tokens, words, d_words, d_x_tm, W, dtable, p=0.0, seed=0, stream_id=0):
    """dtable[V, W] (fp32, accumulated with atomics) += (d_words + d_x_tm^T) * tanh'(words) * mask."""
    B, L, Wp = words.shape
    assert dtable.dtype == F32 and dtable.is_contiguous() and dtable.shape[1] == W
    for t in (d_words, d_x_tm):
        assert t is None or (t.dtype == words.dtype and t.is_contiguous() and t.numel() == words.numel())
    _lib.check(_v("embed_bwd", words)(_ptr(tokens), _ptr(words), _ptr(d_words), _ptr(d_x_tm), B, L, W, Wp, _ptr(dtable), float(p),
                              int(seed), int(stream_id), _stream()), "dvgr_embed_bwd")
    return dtable


def view_attn_fwd_multi(hidden, z, x, w2, want_embed=True):
    """hidden, z: [S, 2, M, D] bf16; x [S, M, D] bf16; w2 [S, D] f32 -> (xnew [S,M,D], embed [S,M,D] | None, beta [S,M,2])."""
    S, _, M, D = z.shape
    assert hidden.is_contiguous() and z.is_contiguous() and x.is_contiguous() and w2.is_contiguous() and w2.dtype == F32
    xnew = torch.empty_like(x)
    embed = torch.empty_like(x) if want_embed else None
    beta = _empty((S, M, 2), F32, x)
    _lib.check(_lib.view_attn_fwd_multi(_ptr(hidden), _ptr(z), _ptr(x), _ptr(w2), M, D, S, _ptr(xnew), _ptr(embed), _ptr(beta),
                                        _stream()), "dvgr_view_attn_fwd_multi")
    return xnew, embed, beta


def view_attn_bwd_multi(dxnew, dembed, hidden, z, w2, beta):
    """-> dz [S,2,M,D], dhid [S,2,M,D] (tanh' applied), dw2 partials [S, blocks, D]."""
    S, _, M, D = z.shape
    assert dxnew.is_contiguous() and (dembed is None or dembed.is_contiguous())
    dz, dhid = torch.empty_like(z), torch.empty_like(hidden)
    blocks = int(_lib.lib.dvgr_view_attn_bwd_blocks(M))
    part = _empty((S, blocks, D), F32, z)
    _lib.check(_lib.view_attn_bwd_multi(_ptr(dxnew), _ptr(dembed), _ptr(hidden), _ptr(z), _ptr(w2), _ptr(beta), M, D, S,
                                        _ptr(dz), _ptr(dhid), _ptr(part), _stream()), "dvgr_view_attn_bwd_multi")
    return dz, dhid, part


def cast_rows_grouped(params, out, out_cols=None, lstm_H=0):
    """Row-concatenated bf16 copy of several fp32 matrices (equal column count) in ONE launch; see cast_rows."""
    C = params[0].shape[1]
    oc = out_cols or C
    n = len(params)
    assert n <= 8 and out.dtype == BF16 and out.stride(1) == 1 and out.shape[1] >= oc
    ins, outs, r = [], [], 0
    lds, rows, cols = (ctypes.c_longlong * n)(), (ctypes.c_int * n)(), (ctypes.c_int * n)()
    for i, p in enumerate(params):
        assert p.dtype == F32 and p.dim() == 2 and p.stride(1) == 1 and p.shape[1] == C
        ins.append(p)
        outs.append(out[r:r + p.shape[0]])
        lds[i], rows[i], cols[i] = p.stride(0), p.shape[0], C
        r += p.shape[0]
    _lib.check(_lib.cast_rows_grouped(_parr(ins), lds, _parr(outs), rows, cols, n, out.stride(0), oc, lstm_H, _stream()),
               "dvgr_cast_rows_grouped")
    return out


def lstm_pack_bias(b_ih, b_hh, H):
    """[D*4H] f32 gate-interleaved b_ih + b_hh of D directions (lists of [4H] tensors) in one launch."""
    D = len(b_ih)
    out = _empty((D * 4 * H,), F32, b_ih[0])
    _lib.check(_lib.lstm_pack_bias(_parr(b_ih), _parr(b_hh), D, H, _ptr(out), _stream()), "dvgr_lstm_pack_bias")
    return out


def lstm_pack_dh(d_seq, nd_seq, d_last, d_last0, S, T, D, H):
    """(dh_seq blocked [T,D,RB,H/8,32,8], dh_last [S, D*H]) from the strided gradients of an encoder's outputs."""
    like = d_seq if d_seq is not None else d_last
    RB, UG = (S + 31) // 32, H // 8
    dh_seq = _empty((T, D, RB, UG, 32, 8), BF16, like)
    dh_last = _empty((S, D * H), BF16, like)
    ld_seq = d_seq.stride(-2) if d_seq is not None else 8
    ld_last = d_last.stride(0) if d_last is not None else 8
    if d_seq is not None:
        assert d_seq.dtype == BF16 and d_seq.stride(-1) == 1 and d_seq.dim() == 3 and d_seq.stride(0) == T * ld_seq
    if d_last is not None:
        assert d_last.dtype == BF16 and d_last.stride(-1) == 1
    _lib.check(_lib.lstm_pack_dh(_ptr(d_seq), ld_seq, nd_seq, _ptr(d_last), ld_last, d_last0, S, T, D, H, _ptr(dh_seq),
                                 _ptr(dh_last), _stream()), "dvgr_lstm_pack_dh")
    return dh_seq, dh_last


def finalize_loss(ce, parts, flags):
    """[4] f32 = (total = ce + sum(parts), common sum, dependence sum, #set flags); total is NaN when a flag is set.
    ce: 1-element f32 tensor; parts: [..., 3] f32 contiguous or None; flags: list of 1-element int32 tensors (<= 16)."""
    out = _empty((4,), F32, ce)
    rows = parts.numel() // 3 if parts is not None else 0
    _lib.check(_lib.finalize_loss(_ptr(ce), _ptr(parts), rows, _parr(flags), len(flags), _ptr(out), _stream()),
               "dvgr_finalize_loss")
    return out


def accuracy_counters(logits, answers, counts, category=None, tokens=None, token_to_cat=None, want_preds=False):
    """counts [n_cat + 1, 2] int64 += (correct, total) per category and overall (last row); see dvgr_accuracy_counters."""
    B, A = logits.shape
    assert logits.dtype == F32 and logits.is_contiguous() and answers.dtype == torch.int64 and counts.dtype == torch.int64
    n_cat = counts.shape[0] - 1
    preds = torch.empty((B,), dtype=torch.int32, device=logits.device) if want_preds else None
    if category is not None:
        assert category.dtype == torch.int64 and category.is_contiguous()
    V = 0
    if tokens is not None:
        assert tokens.dtype == torch.int64 and tokens.stride(-1) == 1 and token_to_cat.dtype == torch.int32
        V = token_to_cat.numel()
    _lib.check(_lib.accuracy_counters(_ptr(logits), _ptr(answers), B, A, _ptr(category), _ptr(tokens),
                                      tokens.stride(0) if tokens is not None else 0, _ptr(token_to_cat), V, n_cat, _ptr(counts),
                                      _ptr(preds), _stream()), "dvgr_accuracy_counters")
    return preds


# ------------------------------------------------------------------------------------- fp32 mode: 3 x bf16 split products
def split3(x, out=None):
    """fp32 [R, C] (last dim contiguous) -> bf16 planes [3, R, Cp] = [lo | hi | hi], Cp = C rounded up to 8."""
    assert x.dtype == F32 and x.dim() == 2 and x.stride(1) == 1
    R, C = x.shape
    Cp = (C + 7) // 8 * 8
    if out is None:
        out = torch.empty((3, R, Cp), dtype=BF16, device=x.device)
    assert out.is_contiguous() and tuple(out.shape) == (3, R, Cp)
    _lib.check(_lib.split3(_ptr(x), x.stride(0), R, C, _ptr(out), Cp, _stream()), "dvgr_split3")
    return out


def gemm3(A3, a_major, B3, b_major, M, N, K, C, batch=1, a_shared=False, b_shared=False, **kw):
    """fp32-accurate product of two split operands (split3 planes, [3, rows, cols]): C (fp32) = act(A B^T + bias) (+ C).
    K is the TRUE reduction length; operands as for gemm() (major 0: [rows, K], major 1: [K, rows]).
    batch > 1: operands are [batch * 3, rows, cols] (the planes of problem b at 3b .. 3b+2; a_shared / b_shared: every problem
    reads the planes of problem 0), C is [batch, M, N] with c_batch given by the caller."""
    assert C.dtype == F32 and A3.shape[0] == (3 if a_shared else 3 * batch) and B3.shape[0] == (3 if b_shared else 3 * batch)
    kin = (K + 63) // 64
    return gemm(A3, a_major, B3, b_major, M, N, 3 * kin * 64, C, k_inner=kin, batch=batch,
                a_c2=[0 if a_shared else 3 * b for b in range(batch)], a_c2_step=[1] * batch,
                b_c2=[2 if b_shared else 3 * b + 2 for b in range(batch)], b_c2_step=[-1] * batch, **kw)
