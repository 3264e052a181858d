/* dualvgr_b200.h — C ABI of libdualvgr_b200.so: the sm_100a kernels behind the DualVGR reasoning core.
 *
 * The reference (NJUPT-MCC/DualVGR-VideoQA) has no FFI layer: its boundary is the PyTorch nn.Module contract of
 * model/models.py (DualVGR, DualVGRUnit_multiple). Each entry point below replaces the stock ATen call sequence of one
 * reference call site (cited per function as <file>:<lines>, paths relative to the reference root) and is what a
 * ctypes / cffi binding on the reference side would bind (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain pointers + extents; every pointer is a DEVICE pointer unless stated otherwise
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream, never allocates device
 *     memory, never synchronises; outputs and workspaces are allocated by the caller
 *   - activations are bf16 (`uint16_t` storage) unless the name says f32; parameters and their gradients are fp32;
 *     bf16 copies of the weights are produced by dvgr_cast_* once per optimizer step
 *   - return value: 0 on success, non-zero on error; dvgr_last_error() returns a thread-local message
 *   - stateless and re-entrant (an internal cache of TMA descriptors is mutex-protected)
 */
#ifndef DUALVGR_B200_H_
#define DUALVGR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVGR_ABI_VERSION 1

const char* dvgr_last_error(void);
int dvgr_abi_version(void);
/* Number of kernels launched by this library in the calling process so far (bench.py reports the delta). */
long long dvgr_launch_count(void);
/* Optional device-resident counter added to every dropout seed (NULL disables). A train step captured in a CUDA graph
 * increments it on the device, so each replay draws fresh Philox masks although the kernel arguments are frozen. */
void dvgr_set_seed_offset(const unsigned long long* dev_ptr);

/* ------------------------------------------------------------------------------------------------------------------
 * GEMM family (tcgen05 + TMEM + TMA).  D[b][m][n] = epi( sum_k A[b][m][k] * B[b][n][k] ), bf16 operands, fp32 accumulate.
 * An operand is described by up to 4 dims, dims[0] contiguous:
 *   major == 0 (K-major):  dims = {K, rows, d2, d3}     the tensor as nn.Linear sees it (x[M,K], W[N,K])
 *   major == 1 (MN-major): dims = {rows, K, d2, d3}     the same storage seen by dgrad / wgrad (no transposed copies)
 * strides are in ELEMENTS (strides[0] must be 1, all others multiples of 8).
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct dvgr_operand {
  const void* ptr;
  int major;
  int ndim;
  long long dims[4];
  long long strides[4];
} dvgr_operand;

enum { DVGR_ACT_NONE = 0, DVGR_ACT_ELU = 1, DVGR_ACT_TANH = 2 };

typedef struct dvgr_gemm_args {
  dvgr_operand A, B;
  int M, N, K, batch;                 /* batch <= 4 */
  int a_c0[4], a_c2[4], a_c3[4];      /* per-batch coordinate offsets into dims 0, 2, 3 of A */
  int b_c0[4], b_c2[4], b_c3[4];
  int k_inner;                        /* MN-major reductions over [segments][rows]: 64-row blocks per segment, 0 = flat */
  int a_c2_step[4], b_c2_step[4];     /* dims-2 coordinate increment per segment */
  /* linear epilogue:  C = act(acc + bias) (+ C when beta)                                  */
  void* C;
  long long ldc, c_batch;             /* elements */
  int out_f32, act, beta;             /* beta: 0 overwrite, 1 C += (read-modify-write), 2 atomic add (fp32 C only) */
  const float* bias;
  long long bias_batch;
  const int* row_map;                 /* optional output-row permutation (wgrad of gate-interleaved LSTM weights) */
  int bn;                             /* N tile: 128, 256, or 0 = choose */
  int max_ctas;                       /* 0 = one CTA per SM */
  int ksplit;                         /* > 1: split the reduction over that many CTAs per tile (needs beta == 2) */
  int* tile_counter;                  /* optional device int, ZERO on entry: the CTAs claim their tiles from it (dynamic
                                         schedule) instead of a static round-robin deal — for long launches that share the
                                         GPU with kernels on other streams (a CTA that starts late just takes fewer tiles) */
} dvgr_gemm_args;

/* Replaces every nn.Linear forward / dgrad / wgrad on the path: model/models.py:46,74 (motion projection),
 * model/GraphNN.py:96 (GAT head projections), model/Attention.py:14-18 (view-attention MLP),
 * model/fusions/fusions.py:420-449 (MFB), model/AnswerDecoder.py:173-200 (read-out, classifier),
 * model/utils.py:68 (QueryAttn.feat_enhance), and the W_ih product of nn.LSTM at model/Preprocessing.py:227. */
int dvgr_gemm(const dvgr_gemm_args* args, void* stream);

/* Several independent weight gradients in ONE persistent launch:  out_i[rows_i][cols_i] += dy_i[M_i][rows_i]^T x_i[M_i][cols_i]
 * (bf16 operands read MN-major, fp32 accumulation into out_i with vector reductions: out_i must hold the value to add to,
 * e.g. a zeroed gradient buffer). The weight-gradient GEMMs of the nn.Linear layers listed under dvgr_gemm are off the
 * backward pass's critical path; queued and flushed together they form one tile stream instead of ~30 latency-bound
 * launches. `probs` is a HOST array; row strides in elements (multiples of 8), pointers 16-byte aligned. */
typedef struct dvgr_wgrad_problem {
  const void* dy;
  long long ld_dy;
  const void* x;
  long long ld_x;
  int M, rows, cols;
  float* out;
  long long ldc;
} dvgr_wgrad_problem;
int dvgr_wgrad_grouped(const dvgr_wgrad_problem* probs, int n, void* stream);

/* Test-only SIMT reference product (fp32 out), arbitrary element strides:  C[m][n] = sum_k A[m*a_rs + k*a_ks] * B[n*b_rs + k*b_ks] */
int dvgr_gemm_reference(const void* A, long long a_rs, long long a_ks, const void* B, long long b_rs, long long b_ks,
                        float* C, long long ldc, int M, int N, int K, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Fused LSTM recurrence (nn.LSTM(2048, 384, bidirectional) at model/Preprocessing.py:201,227; also usable for the two
 * question BiLSTMs at model/Preprocessing.py:97-101).  One call = one time step of BOTH directions:
 *   recurrent GEMM h_{s} W_hh^T on tensor cores, cell update in the epilogue.
 * Layouts (H hidden, S sequences, T steps, D = ndir directions, gate columns interleaved 4*j + {i,f,g,o}):
 *   gates  [T][S][D*4H] bf16 : in = x_t W_ih^T + b (from dvgr_gemm), out = activated gates (kept for backward);
 *                              after dvgr_lstm_step_bwd it holds the pre-activation gate gradients
 *   h_hist [D][T+1][S][H] bf16, c_hist [D][T+1][S][H] f32 : slot 0 = initial state (zeros), slot s+1 = state after step s
 *   whh    [D][4H][H] bf16 (rows interleaved like the gate columns)
 *   direction d processes time t = s (d even) or T-1-s (d odd) at step s; up to 4 directions per call (two BiLSTMs)
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct dvgr_lstm_args {
  int S, H, T, ndir, s;
  void* gates;
  const void* whh;
  void* h_hist;
  float* c_hist;
  void* h_last;             /* optional [S][h_last_ld] bf16: final hidden of direction d at column d*H (written at s = T-1) */
  long long h_last_ld;
  const int* seq_len;       /* optional [S] int32: steps with t >= len carry the state and emit zeros */
  void* seq_out;            /* optional [S][T][seq_out_ld] bf16 per-step hidden (column d*H) */
  long long seq_out_ld;
  /* backward only */
  float* dc;                /* [D][S][H] f32 running cell-state gradient, zero before the first backward step */
  const void* dh_last;      /* [S][dh_last_ld] bf16 gradient of h_last (used at s = T-1) */
  long long dh_last_ld;
  const void* dh_seq;       /* optional [S][T][seq_out_ld] bf16 gradient of seq_out */
  float* dh_carry;          /* [D][S][H] f32, zero before the first backward step; required with seq_len */
  int max_ctas;             /* whole-sequence kernels only: cap on the persistent grid (0 = one CTA per SM). Their tiles are
                               claimed dynamically, so a smaller grid just leaves SMs to kernels on other streams (a concurrent
                               NCCL all-reduce, the other encoder's recurrence) */
} dvgr_lstm_args;

int dvgr_lstm_step_fwd(const dvgr_lstm_args* args, void* stream);
/* Backward of step s; must be called for s = T-1, T-2, ..., 0. */
int dvgr_lstm_step_bwd(const dvgr_lstm_args* args, void* stream);

/* Whole-sequence forward of the same recurrence in ONE persistent launch, with the input projection fused in
 * (model/Preprocessing.py:227 `self.encoder(...)` = nn.LSTM forward; :97-101,112-123 for the question BiLSTMs):
 *   per (step, direction, 128-sequence block, 256-gate-column block) tile: x_t W_ih^T + h_s W_hh^T on tensor cores
 *   (K = K1 + H in one accumulator), then bias + cell update in the epilogue. The [T][S][D*4H] pre-activations never
 *   reach HBM. Steps are chained inside the launch by per-(direction, block) completion counters, not by kernel boundaries.
 *   x    [T][S][x_ld] bf16 time-major input (K1 valid columns, K1 % 8 == 0)
 *   wih  [D*4H][wih_ld] bf16, rows gate-interleaved like whh (dvgr_cast_rows with lstm_H)
 *   bias [D*4H] f32 = b_ih + b_hh, gate-interleaved
 *   sync [dvgr_lstm_seq_sync_words(S, D)] int32, ZERO on entry: per-(direction, block) completion counters, the counter
 *        the CTAs claim their tiles from (dynamic schedule: no CTA ever waits on a tile that a non-resident CTA owns, so the
 *        launch is safe next to concurrent kernels on other streams), and LAST a sticky error flag (stays 0 unless a
 *        dependency poll timed out, which only a protocol violation can cause)
 * BLOCKED LAYOUT. The tensors that only the cell epilogues of the two whole-sequence calls touch are stored as
 * [piece][row] warp tiles (32 sequences x 8 hidden units; RB = ceil(S / 32) row blocks), so that every warp access is 512
 * contiguous bytes instead of 32 scattered 16-byte pieces:
 *   lstm.gates  [T][D][RB][H/8][4][32][8] bf16  ACTIVATED gates out (piece q = units 2q, 2q+1 x {i,f,g,o})
 *   lstm.c_hist [D][T+1][RB][H/8][2][32][4] f32 (piece q = units 4q..4q+3); slot 0 = initial state (zeros)
 *   lstm.dc     [D][RB][H/8][2][32][4] f32      (backward)
 * h_hist keeps the standard [D][T+1][S][H] layout (it is a TMA / wgrad operand). `lstm.s` is ignored. 4H % 256 == 0. */
typedef struct dvgr_lstm_seq_args {
  dvgr_lstm_args lstm;
  const void* x;
  long long x_ld;
  int K1;
  const void* wih;
  long long wih_ld;
  const float* bias;
  int* sync;
} dvgr_lstm_seq_args;
int dvgr_lstm_seq_sync_words(int S, int ndir);
int dvgr_lstm_seq_fwd(const dvgr_lstm_seq_args* args, void* stream);
/* Whole backward pass of the recurrence (autograd of nn.LSTM at model/Preprocessing.py:227 / :97-101): the cell backward
 * of step T-1 (elementwise) followed by ONE persistent launch for steps T-2 ... 0 (dh_s = dgates_{s+1} W_hh on tensor
 * cores, cell backward in the epilogue, steps chained by completion counters). Consumes the BLOCKED gates / c_hist of
 * dvgr_lstm_seq_fwd and a blocked, zeroed dc; writes the pre-activation gate gradients to `dgates` [T][S][D*4H] bf16
 * (standard layout: the operand of the W_ih / W_hh / bias gradients). With seq_len: dh_carry is blocked like dc
 * ([D][RB][H/8][2][32][4] f32, zeroed) and dh_seq is blocked [T][D][RB][H/8][32][8] bf16. `sync` as for
 * dvgr_lstm_seq_fwd (zero on entry); `args->s` is ignored. */
int dvgr_lstm_seq_bwd(const dvgr_lstm_args* args, void* dgates, int* sync, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Video-based multi-view graph attention (punishGAT): model/GraphNN.py:95-113 for all heads of a graph, plus the head
 * concat and the attention / output dropouts of :107,:175-177. Up to 4 graphs per launch (acGCN, appearance_GCN, mcGCN,
 * motion_GCN of one DualVGR unit, model/models.py:151-158); one CTA per (video, graph), node block staged in shared memory.
 *   wh    [B*N][ld_wh] bf16 : W_k x + b_k of the graph's heads, concatenated along columns (from dvgr_gemm)
 *   gate  [B][N] f32        : QueryPunish gate of the stream (applied to the values only, after the logits)
 *   avec  [heads][2*Dh+1] f32 : a_k[:Dh] | a_k[Dh:] | c_k   (attention_k.a.weight, attention_k.a.bias)
 *   adj   [N][N] f32        : edge iff adj > 0 (a fully masked row yields uniform attention, as in the reference)
 *   out   [B*N][ld_out] bf16
 * Backward additionally needs out (forward result), dout, and writes dwh, dgate [B][N] (zeroed inside the call: the
 * tensor-core path adds the partial sums of its two head-pair CTAs), davec partials [B][heads][2*Dh+1] (sum over B with
 * dvgr_colsum). D = 768 with 4 heads and N <= 32 (forward: <= 64) take the mma.sync fast path; DVGR_GAT_FAST=0 disables it.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct dvgr_gat_graph {
  const void* wh;
  const float* gate;
  const float* avec;
  void* out;
  float* out_f32;           /* optional dense [B*N][D] f32 copy of out (what the auxiliary losses read) */
  const void* dout;
  const float* dout_f32;    /* optional extra gradient on the f32 copy */
  void* dwh;
  float* dgate;
  float* davec;
  unsigned int drop_stream;
} dvgr_gat_graph;

typedef struct dvgr_gat_args {
  dvgr_gat_graph graphs[4];
  int n_graphs;
  int B, N, D, heads;
  long long ld_wh, ld_out;
  const float* adj;
  float slope;              /* LeakyReLU slope, 0.01 in the reference (model/models.py:95) */
  float p_att, p_out;       /* dropout probabilities; 0 = eval / parity mode */
  unsigned long long seed;
} dvgr_gat_args;

int dvgr_gat_attn_fwd(const dvgr_gat_args* args, void* stream);
int dvgr_gat_attn_bwd(const dvgr_gat_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Query Punishment Module (model/utils.py:60-105).
 * dvgr_qattn_fwd: QueryAttn.forward tail (model/utils.py:68-84) given y = feat_enhance(dynamic_q) [B][L][D] bf16 from
 *   dvgr_gemm: L2-normalise, fc score, softmax over ALL L positions, question_len mask (no per-sample host loop),
 *   renormalise (eps 1e-5), q_c = alpha . words.   Saves alpha, nrm, prob [B][L] and ssum [B] for backward.
 *   words [B][L][ld_w] bf16; qc [B][ld_qc] bf16 (columns W..ld_qc-1 zeroed: it is the K-padded A operand of the
 *   QueryPunish.query_weight GEMM, model/utils.py:100).
 * dvgr_gate_fwd: QueryPunish.forward tail (model/utils.py:101-103): gate[b][n] = sigmoid(X[b][n] . query[b]) for the
 *   appearance (x0 / columns 0..D-1 of query) and motion (x1 / columns D..2D-1) streams in one launch.
 * ------------------------------------------------------------------------------------------------------------------ */
int dvgr_qattn_fwd(const void* y, const float* wf, const float* cf, const int* qlen, const void* words, long long ld_w,
                   int B, int L, int D, int W, float* alpha, float* nrm, float* prob, float* ssum, void* qc,
                   long long ld_qc, void* stream);
/* dy [B][L][D] bf16, dwords [B][L][ld_w] bf16 (+= when accumulate_dwords), dwf_part [B][D], dcf_part [B] (sum over B). */
int dvgr_qattn_bwd(const void* dqc, long long ld_qc, const void* y, const float* wf, const int* qlen, const void* words,
                   long long ld_w, int B, int L, int D, int W, const float* alpha, const float* nrm, const float* prob,
                   const float* ssum, void* dy, void* dwords, int accumulate_dwords, float* dwf_part, float* dcf_part,
                   void* stream);
int dvgr_gate_fwd(const void* x0, const void* x1, const void* query, long long ld_q, int B, int N, int D, float* gate0,
                  float* gate1, void* stream);
/* dgate of stream s = dg{s}a (+ dg{s}b: the two graphs sharing the gate, model/models.py:151-158).
 * dx{s} [B][N][D] bf16 is ACCUMULATED into; dquery [B][ld_q] bf16 is written. */
int dvgr_gate_bwd(const void* x0, const void* x1, const void* query, long long ld_q, int B, int N, int D,
                  const float* gate0, const float* gate1, const float* dg0a, const float* dg0b, const float* dg1a,
                  const float* dg1b, void* dx0, void* dx1, void* dquery, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Two-view attention + residual: AttentionSFGCN.forward (model/Attention.py:20-23) on the [common, specific] stack of
 * model/models.py:163-166 and the residual add of :168-169.
 *   hidden [2][M][D] bf16 = tanh(project.0(z)) from dvgr_gemm (tanh epilogue); z [2][M][D] bf16; x [M][D] bf16
 *   xnew = x + sum_v beta_v z_v ; embed (optional) = sum_v beta_v z_v ; beta [M][2] f32
 * Backward: dxnew is also the gradient of x (residual) — the caller keeps accumulating into that buffer.
 *   dz [2][M][D], dhid [2][M][D] (tanh' applied: feeds the project.0 dgrad/wgrad), dw2_part [dvgr_view_attn_bwd_blocks(M)][D]
 * ------------------------------------------------------------------------------------------------------------------ */
int dvgr_view_attn_fwd(const void* hidden, const void* z, const void* x, const float* w2, long long M, int D, void* xnew,
                       void* embed, float* beta, void* stream);
int dvgr_view_attn_bwd_blocks(long long M);
/* Both input streams (appearance, motion) of a unit in one launch: every operand of dvgr_view_attn_fwd / _bwd gains a leading
 * [n_streams] dimension (hidden, z, dz, dhid: [S][2][M][D]; x, xnew, embed, dxnew, dembed: [S][M][D]; w2 [S][D]; beta [S][M][2];
 * dw2_part [S][blocks][D]). */
int dvgr_view_attn_fwd_multi(const void* hidden, const void* z, const void* x, const float* w2, long long M, int D,
                             int n_streams, void* xnew, void* embed, float* beta, void* stream);
int dvgr_view_attn_bwd_multi(const void* dxnew, const void* dembed_ext, const void* hidden, const void* z, const float* w2,
                             const float* beta, long long M, int D, int n_streams, void* dz, void* dhid, float* dw2_part,
                             void* stream);
int dvgr_view_attn_bwd(const void* dxnew, const void* dembed_ext, const void* hidden, const void* z, const float* w2,
                       const float* beta, long long M, int D, void* dz, void* dhid, float* dw2_part, void* stream);

/* MFB pair-sum (model/fusions/fusions.py:433-441): z[M][mm2/2] = pairsum(x0 * x1), x0/x1 [M][mm2] already ELU'd. */
int dvgr_mfb_fwd(const void* x0, const void* x1, void* z, long long M, int mm2, void* stream);
int dvgr_mfb_bwd(const void* dz, const void* x0, const void* x1, void* d0, void* d1, long long M, int mm2, void* stream);

/* Attention read-out (model/AnswerDecoder.py:176-180): alpha = softmax_n(w . u_n + c), pooled[b] = sum_n alpha_n v_n,
 * u = ELU(v_proj(v)) from dvgr_gemm; pooled is written with row stride ld_p (left half of the classifier input). */
int dvgr_readout_fwd(const void* v, const void* u, const float* w, const float* c, int B, int N, int D, float* alpha,
                     void* pooled, long long ld_p, void* stream);
int dvgr_readout_bwd(const void* dpooled, long long ld_p, const void* v, const void* u, const float* w,
                     const float* alpha, int B, int N, int D, void* dv, void* du, float* dw_part, float* dc_part,
                     void* stream);

/* BatchNorm1d of the classifier (model/AnswerDecoder.py:193). x [B][D] is f32 (x_is_f32, the precise path: centring
 * a bf16-rounded input amplifies its rounding error by |x|/std) or bf16; y and dy are bf16; dx has x's type. */
int dvgr_bn_fwd(const void* x, int x_is_f32, int B, int D, const float* gamma, const float* beta, float* run_mean,
                float* run_var, int training, float momentum, float eps, void* y, float* mean_out, float* rstd_out,
                void* stream);
int dvgr_bn_bwd(const void* dy, const void* x, int x_is_f32, int B, int D, const float* gamma, const float* mean,
                const float* rstd, int training, void* dx, float* dgamma, float* dbeta, void* stream);
/* Synchronised BatchNorm over a data-parallel group (the classifier's nn.BatchNorm1d sees the GLOBAL batch, as the reference
 * does on one GPU): dvgr_bn_stats writes the local per-column (sum, sum of squares) [2][D]; the caller all-reduces them and
 * passes them as ext_stats with the global row count Btot. Backward: a first call with stats_only = 1 writes the LOCAL
 * (sum dy -> dbeta, sum dy*xhat -> dgamma) and stops; the caller all-reduces [dbeta | dgamma] and passes them as ext_sums
 * [2][D] to a second call (dgamma / dbeta may then be null). ext_* == null reproduces dvgr_bn_fwd / dvgr_bn_bwd. */
int dvgr_bn_stats(const void* x, int x_is_f32, int B, int D, float* out, void* stream);
int dvgr_bn_fwd_ex(const void* x, int x_is_f32, int B, int D, const float* gamma, const float* beta, float* run_mean,
                   float* run_var, int training, float momentum, float eps, void* y, float* mean_out, float* rstd_out,
                   const float* ext_stats, int Btot, void* stream);
int dvgr_bn_bwd_ex(const void* dy, const void* x, int x_is_f32, int B, int D, const float* gamma, const float* mean,
                   const float* rstd, int training, void* dx, float* dgamma, float* dbeta, const float* ext_sums, int Btot,
                   int stats_only, void* stream);

/* nn.CrossEntropyLoss (train.py:121,146) value + gradient: loss_part[b] (sum = mean CE), dlogits [B][ld_d] bf16 =
 * (softmax - onehot) * scale / B with zeroed padding columns, correct[b] = argmax == answer (train.py:352-356). */
int dvgr_cross_entropy(const float* logits, const long long* answers, int B, int A, float scale, float* loss_part,
                       void* dlogits, long long ld_d, int* correct, void* stream);
/* Same with the gradient written as fp32 when grad_is_f32 (the dtype of the logits: what autograd hands to their producer). */
int dvgr_cross_entropy_ex(const float* logits, const long long* answers, int B, int A, float scale, float* loss_part,
                          void* dlogits, int grad_is_f32, long long ld_d, int* correct, void* stream);
/* Validation bookkeeping on the device (validate.py:59-134: argmax, agreeings, per-question-type / per-category accuracy —
 * Python loops with a host sync per sample in the reference): counts [n_cat + 1][2] int64 += {correct, total} per category,
 * row n_cat = all samples. The category of sample b is category[b] (SVQA: question_categories, validate.py:44) or, when
 * category is null, token_to_cat[tokens[b][0]] (MSVD / MSRVTT: first question word -> what / who / how / when / where,
 * validate.py:66-80; -1 = none). preds (optional) [B] int32 receives the argmax (first index on ties). */
int dvgr_accuracy_counters(const float* logits, const long long* answers, int B, int A, const long long* category,
                           const long long* tokens, long long ld_tok, const int* token_to_cat, int V, int n_cat,
                           long long* counts, int* preds, void* stream);

/* Auxiliary losses (utils.py:10-31), value and gradient fused; up to 4 (x, y) pairs per call (one DualVGR unit needs 3:
 * common(com_app, com_mot), HSIC(aq, com_app), HSIC(mq, com_mot) — train.py:148-154). x, y, dx, dy are [B][N][D] f32.
 * mode 0: coef * sum_ij (G_x - G_y)^2 (common_loss numerator) ; mode 1: coef * tr(R K_x R K_y) (HSIC).
 * loss_part[b][loss_col] (row stride loss_ld) receives the per-video value; accumulate_{x,y}: 0 write, 1 add in place,
 * 2 atomicAdd into a caller-zeroed buffer (for a tensor that is an operand of two pairs of the same call).
 * gram_ws: dvgr_pair_loss_workspace(...) floats. */
typedef struct dvgr_pair_job {
  const float* x;
  const float* y;
  float* dx;
  float* dy;
  float* loss_part;
  int loss_col, loss_ld;
  int mode;
  int accumulate_x, accumulate_y;
  float coef;
} dvgr_pair_job;
long long dvgr_pair_loss_workspace(int n_jobs, int B, int N, int D);
int dvgr_pair_loss_multi(const dvgr_pair_job* jobs, int n_jobs, int B, int N, int D, float* gram_ws, void* stream);
/* The three auxiliary terms of ONE DualVGR unit in a tensor-centric form (train.py:148-154 for one layer):
 *   coef_com * sum_ij (G_ca - G_cm)^2  +  coef_dep * (HSIC(aq, ca) + HSIC(mq, cm)),
 * value and the COMPLETE gradients of the four [B][N][D] f32 operands in two launches (each operand tile is loaded once
 * per pass, every gradient is written with plain stores: no atomics, no pre-zeroed buffers). loss_part [B][3] receives the
 * per-video coef-scaled (common, HSIC_app, HSIC_motion); gradients may be NULL (value only);
 * gram_ws: dvgr_aux_loss_workspace(B, N, D) floats. */
long long dvgr_aux_loss_workspace(int B, int N, int D);
int dvgr_aux_loss_unit(const float* ca, const float* cm, const float* aq, const float* mq, float coef_com, float coef_dep,
                       int B, int N, int D, float* d_ca, float* d_cm, float* d_aq, float* d_mq, float* loss_part,
                       float* gram_ws, void* stream);
/* precise != 0: the Gram products run on error-compensated 3 x TF32 (fp32-grade; fp32 mode) instead of plain TF32. */
int dvgr_aux_loss_unit_ex(const float* ca, const float* cm, const float* aq, const float* mq, float coef_com, float coef_dep,
                       int B, int N, int D, float* d_ca, float* d_cm, float* d_aq, float* d_mq, float* loss_part,
                       float* gram_ws, int precise, void* stream);

/* Streaming helpers.
 * dvgr_prep_features: model/Preprocessing.py:220-223 — tanh(dropout(x)), fp32 -> bf16, [S][T][C] -> [T][S][C] in one pass.
 * dvgr_cast_rows: fp32 parameter -> bf16 GEMM operand (zero-padded columns; lstm_H > 0 interleaves LSTM gate rows).
 * dvgr_dropout: out = in * mask/(1-p) (its own backward). dvgr_act_bwd: out (+)= dy * mask * act'(y).
 * dvgr_colsum: out[C] (+)= scale * sum_r in[r][c] (bias gradients, per-video partial reductions); deterministic. */
int dvgr_prep_features(const float* in, void* out, long long S, int T, int C, int do_tanh, int time_major, float p,
                       unsigned long long seed, unsigned int drop_stream, void* stream);
/* Same pass for features that are stored / shipped as bf16 (in_is_bf16 = 1): halves the 713 MB per step that the fp32
 * features of the reference's DataLoader (DataLoader.py:61-84) put on the host link (SURVEY.md §8f.3). */
int dvgr_prep_features_ex(const void* in, int in_is_bf16, void* out, long long S, int T, int C, int do_tanh,
                          int time_major, float p, unsigned long long seed, unsigned int drop_stream, void* stream);
/* The same pass over a batch gathered from a device-resident feature store: store [V][N][T][C] (fp32, or bf16 when
 * store_is_bf16), rows [B] int32 device -> out exactly as dvgr_prep_features_ex(store[rows], S = B*N, ...) writes it (same
 * layout, same dropout mask). Replaces the per-sample HDF5 reads of DataLoader.py:61-84 and the host-to-device copy of the
 * batch in front of Preprocessing.py:220-223 (appearance: T = 16, time_major, do_tanh) and models.py:74 (motion: T = 1).
 * A row outside [0, V) is not read: its output rows are zero and *err (device int32, sticky: never cleared here) is set to 1. */
int dvgr_prep_features_gather(const void* store, int store_is_bf16, long long V, int N, const int* rows, int B, void* out,
                              int T, int C, int do_tanh, int time_major, float p, unsigned long long seed,
                              unsigned int drop_stream, int* err, void* stream);
int dvgr_cast_rows(const float* in, long long ld_in, void* out, long long ld_out, int rows, int cols, int out_cols,
                   int lstm_H, void* stream);
/* n (<= 8) dvgr_cast_rows problems sharing ld_out / out_cols / lstm_H in one launch: the bf16 (gate-interleaved) copies of
 * all W_ih or W_hh matrices of an encoder written into one row-concatenated operand. HOST arrays. */
int dvgr_cast_rows_grouped(const float* const* in, const long long* ld_in, void* const* out, const int* rows, const int* cols,
                           int n, long long ld_out, int out_cols, int lstm_H, void* stream);
/* out[d][4j + g] = b_ih[d][g*H + j] + b_hh[d][g*H + j]: the gate-interleaved bias operand of dvgr_lstm_seq_fwd for all
 * directions (nn.LSTM keeps two bias vectors per direction, model/Preprocessing.py:97-101,202). HOST pointer arrays. */
int dvgr_lstm_pack_bias(const float* const* b_ih, const float* const* b_hh, int ndir, int H, float* out, void* stream);
/* Packs the gradients arriving at an LSTM encoder for dvgr_lstm_seq_bwd: d_seq [S][T][ld_seq] bf16 (per-step outputs of
 * directions 0..nd_seq-1, may be null) -> dh_seq blocked [T][D][RB][H/8][32][8]; d_last [S][ld_last] bf16 (final states of
 * directions d_last0..D-1, may be null) -> dh_last [S][D*H]; everything else zero. */
int dvgr_lstm_pack_dh(const void* d_seq, long long ld_seq, int nd_seq, const void* d_last, long long ld_last, int d_last0,
                      int S, int T, int D, int H, void* dh_seq, void* dh_last, void* stream);
/* fp32 mode (1e-4 parity with the reference's fp32 path): an fp32 matrix [rows][cols] (row stride ld_in) as three bf16 planes
 * out [3][rows][ld_out] = [lo | hi | hi], x = hi + lo (16 mantissa bits; ld_out % 8 == 0, padding columns zero). dvgr_gemm
 * multiplies two such operands to fp32 accuracy in ONE launch: describe them as 3-D / 4-D operands with the plane on dims[2],
 * K = 3 * k_inner * 64, k_inner = ceil(true reduction length / 64), A: a_c2 = 0, a_c2_step = +1, B: b_c2 = 2, b_c2_step = -1
 * (a_lo b_hi + a_hi b_hi + a_hi b_lo), out_f32 = 1. Works for K-major and MN-major operands (forward, dgrad, wgrad). */
int dvgr_split3(const float* in, long long ld_in, int rows, int cols, void* out, long long ld_out, void* stream);
int dvgr_dropout(const void* in, void* out, long long n, float p, unsigned long long seed, unsigned int drop_stream,
                 void* stream);
int dvgr_act_bwd(const void* dy, const void* y, void* out, long long n, int act, int accumulate, float p,
                 unsigned long long seed, unsigned int drop_stream, void* stream);
int dvgr_add(void* a, const void* b, long long n, void* stream);
/* The input dropouts of up to 4 punishGATs in one launch (model/GraphNN.py:175: every punishGAT call drops its own copy of
 * the stream it reads): out[i] = in[i] * mask(seed, drop_streams[i]); in / out / drop_streams are HOST arrays of n_copies. */
int dvgr_dropout_multi(const void* const* in, void* const* out, const unsigned int* drop_streams, int n_copies, long long n,
                       float p, unsigned long long seed, void* stream);
/* Backward of those copies merged with the gradient that bypasses the graphs (residual, model/models.py:168-169):
 *   out[s] = base[s] + sum_{j < per_stream} mask(drop_streams[s*per_stream + j]) * dxt[s*per_stream + j],  s < n_streams <= 2.
 * dxt: n_streams*per_stream (<= 4) pointers, base (entries may be null) / out: n_streams pointers; all HOST arrays. */
int dvgr_gat_input_bwd(const void* const* dxt, const unsigned int* drop_streams, int n_streams, int per_stream,
                       const void* const* base, void* const* out, long long n, float p, unsigned long long seed, void* stream);
/* Question-word prologue (model/Preprocessing.py:109-111): words = tanh(dropout(encoder_embed[tokens])) in one pass, written
 * as words [B][L][Wp] bf16 and time-major x_tm [L][B][Wp] bf16 (word dim zero-padded to Wp, Wp % 8 == 0). tokens int64.
 * Backward: dtable[tok] += (d_words[b][l] + d_x_tm[l][b]) * (1 - words^2) * mask (fp32 atomics; either gradient may be null). */
int dvgr_embed_fwd(const long long* tokens, const float* table, int B, int L, int W, int Wp, void* words, void* x_tm,
                   float p, unsigned long long seed, unsigned int drop_stream, void* stream);
int dvgr_embed_bwd(const long long* tokens, const void* words, const void* d_words, const void* d_x_tm, int B, int L, int W,
                   int Wp, float* dtable, float p, unsigned long long seed, unsigned int drop_stream, void* stream);
/* Several column sums in one launch: out_i[C_i] += sum_r in_i[r][c] (always accumulating; fp32 atomics across row
 * chunks). The bias gradients of the nn.Linear layers, queued during backward and flushed once per train step. */
typedef struct dvgr_colsum_problem {
  const void* in;
  int in_is_f32;
  long long ld, R;
  int C;
  float* out;
  int perm_H;     /* > 0 (C == 4 * perm_H): input column 4*j + g lands at out[g * perm_H + j] — the bias gradient of a
                     gate-interleaved LSTM direction written back in nn.LSTM's i|f|g|o order */
  float* out2;    /* optional second target receiving the same sums (bias_ih and bias_hh of nn.LSTM share one gradient) */
} dvgr_colsum_problem;
int dvgr_colsum_grouped(const dvgr_colsum_problem* probs, int n, void* stream);
/* dst[i] (+)= src[i] for a HOST array of small f32 segments, 128 per launch. accumulate = 1: adds the gradients of the many
 * tiny parameters of a unit (per-head attention vectors / biases) into their bound .grad views in one launch instead of
 * one elementwise launch per parameter (what autograd's AccumulateGrad does); accumulate = 0: gathers those parameters
 * into the packed avec / bias operands of dvgr_gat_attn_* (model/GraphNN.py:88-93) instead of ~25 torch.cat launches. */
typedef struct dvgr_seg {
  float* dst;
  const float* src;
  int n;
} dvgr_seg;
int dvgr_scatter(const dvgr_seg* segs, int n_segs, int accumulate, void* stream);
long long dvgr_colsum_workspace(long long R, int C);
int dvgr_colsum(const void* in, int in_is_f32, long long ld, long long R, int C, float* workspace, float* out,
                int accumulate, float scale, void* stream);
/* `batch` independent reductions in one launch pair: in + b * in_batch (elements) -> out + b * out_batch; workspace:
 * batch * dvgr_colsum_workspace(R, C) floats. (Per-graph bias gradients and attention-vector partials of a GAT layer.) */
int dvgr_colsum_batched(const void* in, int in_is_f32, long long ld, long long in_batch, long long R, int C, int batch,
                        float* workspace, float* out, long long out_batch, int accumulate, float scale, void* stream);

/* Flat-buffer optimizer (train.py:85,158-159): sum of squares for clip_grad_norm_(12), then Adam with the clip folded in. */
int dvgr_sumsq_blocks(void);
int dvgr_sumsq(const float* g, long long n, float* partial_ws, float* out, void* stream);
int dvgr_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float max_norm, const float* norm_sq,
                   float grad_scale, const int* step_dev /* optional device step counter, overrides `step` */,
                   void* bf16_shadow /* optional [n] bf16 copy of the updated parameters (next step's GEMM operands) */,
                   void* stream);

/* End-of-step bookkeeping (train.py:154,160-176): out[0] = ce + column sums of parts [rows][3] (the coef-scaled auxiliary
 * loss partials written by dvgr_aux_loss_unit), out[1] = common-loss sum, out[2] = dependence-loss sum, out[3] = number of
 * non-zero words among `flags` (HOST array of n_flags <= 16 device pointers: the sticky error words of this step's
 * dvgr_lstm_seq_* launches). If any flag is set out[0] is NaN: a broken dependency chain can never train silently. */
int dvgr_finalize_loss(const float* ce, const float* parts, int rows, const int* const* flags, int n_flags, float* out,
                       void* stream);

/* ======================================================================================================================
 * fp32 mode (north_star: "within 1e-4 relative error in fp32"). The streaming kernel families above are compiled a second
 * time with fp32 activations (csrc/act.cuh: act_t = float) and exported under the suffix _f32: IDENTICAL signatures, every
 * activation pointer documented as bf16 above is a float pointer here (row strides stay in elements). GEMM-shaped work in
 * fp32 mode runs on the same tcgen05 kernel through three bf16 planes per operand (dvgr_split3 + the k_inner plane
 * segmentation of dvgr_gemm: a_lo b_hi + a_hi b_hi + a_hi b_lo, < 2e-5 of the float64 product); the recurrent cells run in
 * dvgr_lstm32_cell_fwd / _bwd below.
 * ====================================================================================================================== */
int dvgr_gat_attn_fwd_f32(const dvgr_gat_args* args, void* stream);
int dvgr_gat_attn_bwd_f32(const dvgr_gat_args* args, void* stream);
int dvgr_qattn_fwd_f32(const void* y, const float* wf, const float* cf, const int* qlen, const void* words, long long ld_w,
                   int B, int L, int D, int W, float* alpha, float* nrm, float* prob, float* ssum, void* qc,
                   long long ld_qc, void* stream);
int dvgr_qattn_bwd_f32(const void* dqc, long long ld_qc, const void* y, const float* wf, const int* qlen, const void* words,
                   long long ld_w, int B, int L, int D, int W, const float* alpha, const float* nrm, const float* prob,
                   const float* ssum, void* dy, void* dwords, int accumulate_dwords, float* dwf_part, float* dcf_part,
                   void* stream);
int dvgr_gate_fwd_f32(const void* x0, const void* x1, const void* query, long long ld_q, int B, int N, int D, float* gate0,
                  float* gate1, void* stream);
int dvgr_gate_bwd_f32(const void* x0, const void* x1, const void* query, long long ld_q, int B, int N, int D,
                  const float* gate0, const float* gate1, const float* dg0a, const float* dg0b, const float* dg1a,
                  const float* dg1b, void* dx0, void* dx1, void* dquery, void* stream);
int dvgr_view_attn_fwd_f32(const void* hidden, const void* z, const void* x, const float* w2, long long M, int D, void* xnew,
                       void* embed, float* beta, void* stream);
int dvgr_view_attn_bwd_f32(const void* dxnew, const void* dembed_ext, const void* hidden, const void* z, const float* w2,
                       const float* beta, long long M, int D, void* dz, void* dhid, float* dw2_part, void* stream);
int dvgr_mfb_fwd_f32(const void* x0, const void* x1, void* z, long long M, int mm2, void* stream);
int dvgr_mfb_bwd_f32(const void* dz, const void* x0, const void* x1, void* d0, void* d1, long long M, int mm2, void* stream);
int dvgr_readout_fwd_f32(const void* v, const void* u, const float* w, const float* c, int B, int N, int D, float* alpha,
                     void* pooled, long long ld_p, void* stream);
int dvgr_readout_bwd_f32(const void* dpooled, long long ld_p, const void* v, const void* u, const float* w,
                     const float* alpha, int B, int N, int D, void* dv, void* du, float* dw_part, float* dc_part,
                     void* stream);
int dvgr_bn_fwd_ex_f32(const void* x, int x_is_f32, int B, int D, const float* gamma, const float* beta, float* run_mean,
                   float* run_var, int training, float momentum, float eps, void* y, float* mean_out, float* rstd_out,
                   const float* ext_stats, int Btot, void* stream);
int dvgr_bn_bwd_ex_f32(const void* dy, const void* x, int x_is_f32, int B, int D, const float* gamma, const float* mean,
                   const float* rstd, int training, void* dx, float* dgamma, float* dbeta, const float* ext_sums, int Btot,
                   int stats_only, void* stream);
int dvgr_prep_features_ex_f32(const void* in, int in_is_bf16, void* out, long long S, int T, int C, int do_tanh,
                          int time_major, float p, unsigned long long seed, unsigned int drop_stream, void* stream);
int dvgr_prep_features_gather_f32(const void* store, int store_is_bf16, long long V, int N, const int* rows, int B, void* out,
                                  int T, int C, int do_tanh, int time_major, float p, unsigned long long seed,
                                  unsigned int drop_stream, int* err, void* stream);
int dvgr_dropout_f32(const void* in, void* out, long long n, float p, unsigned long long seed, unsigned int drop_stream,
                 void* stream);
int dvgr_act_bwd_f32(const void* dy, const void* y, void* out, long long n, int act, int accumulate, float p,
                 unsigned long long seed, unsigned int drop_stream, void* stream);
int dvgr_add_f32(void* a, const void* b, long long n, void* stream);
int dvgr_embed_fwd_f32(const long long* tokens, const float* table, int B, int L, int W, int Wp, void* words, void* x_tm,
                   float p, unsigned long long seed, unsigned int drop_stream, void* stream);
int dvgr_embed_bwd_f32(const long long* tokens, const void* words, const void* d_words, const void* d_x_tm, int B, int L, int W,
                   int Wp, float* dtable, float p, unsigned long long seed, unsigned int drop_stream, void* stream);

/* fp32 recurrent cell (csrc/lstm32.cu), one launch per time step s of all `ndir` directions (odd directions run backwards:
 * time t = T-1-s). nn.LSTM gate order (i|f|g|o blocks of H). Replaces the cuDNN cell of nn.LSTM for fp32 mode
 * (reference model/Preprocessing.py:97-101,202).
 *   gates        [T][S][ndir*4H] f32: x W_ih^T + b_ih + b_hh on entry; forward overwrites the step's rows with the ACTIVATED
 *                gates, backward writes the pre-activation gate gradients to `dgates` (or over them when dgates is NULL)
 *   rec          [ndir][S][4H] f32: h_{prev} W_hh^T of this step (unused at s == 0)
 *   h            [ndir][S][H] f32 running state; h_planes [ndir][3][S][H] bf16 split of the new state (next step's operand)
 *   c_hist       [T+1][ndir][S][H] f32 by step (slot s in, slot s+1 out; slot 0 is never read)
 *   hprev_t      [ndir][T][S][H] f32: the state BEFORE time t (operand of the W_hh gradient)
 *   seq_out      optional [S][T][seq_out_ld]: h_t at valid positions, 0 at padded ones; h_last [S][h_last_ld] (written at the
 *                last step: the state after the last VALID position, like a packed sequence)
 *   seq_len      optional [S] int32
 * backward: dh / dc [ndir][S][H] f32 running gradients (dh is re-initialised with the part that by-passes the gates; the
 * caller then accumulates dgates W_hh into it), dgate_planes [ndir][3][S][4H] bf16, dh_last [S][dh_last_ld], dh_seq
 * [S][T][dh_seq_ld] (optional). */
typedef struct dvgr_lstm32_args {
  int S, H, T, ndir, s;
  float* gates;
  const float* rec;
  float* h;
  float* c_hist;
  void* h_planes;
  float* hprev_t;
  float* seq_out;
  long long seq_out_ld;
  float* h_last;
  long long h_last_ld;
  const int* seq_len;
  float* dh;
  float* dc;
  void* dgate_planes;
  const float* dh_last;
  long long dh_last_ld;
  const float* dh_seq;
  long long dh_seq_ld;
  float* dgates; /* backward: where the gate gradients go ([T][S][ndir*4H]); NULL = over the activated gates */
} dvgr_lstm32_args;
int dvgr_lstm32_cell_fwd(const dvgr_lstm32_args* args, void* stream);
int dvgr_lstm32_cell_bwd(const dvgr_lstm32_args* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DUALVGR_B200_H_ */
