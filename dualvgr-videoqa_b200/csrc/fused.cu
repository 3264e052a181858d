// Memory-bound fused kernels of the DualVGR unit tail: two-view attention + residual, MFB pair-sum, attention
// read-out, BatchNorm1d, cross-entropy, plus the streaming helpers (feature prologue, weight casts, dropout, ELU
// backward, column sums). Each is a single pass over its operands with 128-bit accesses and warp-shuffle reductions.
#include <cuda_bf16.h>

#include "act.cuh"
#include "capi_internal.h"
#include "ptx.cuh"
#include "rng.cuh"

// (compiled twice, see act.cuh: `bf16` below is the build's activation storage type — __nv_bfloat16, or float in the
//  -DDVGR_F32 build whose entry points carry the suffix _f32; types that must be bf16 in BOTH builds are spelled out)
namespace dvgr {
namespace DVGR_VNS {

typedef act_t bf16;

__device__ __forceinline__ void load8(const bf16* p, float (&f)[8]) { act::ld8(p, f); }
__device__ __forceinline__ void load8g(const __nv_bfloat16* p, float (&f)[8]) { act::ld8(p, f); }
__device__ __forceinline__ void load8g(const float* p, float (&f)[8]) { act::ld8(p, f); }
__device__ __forceinline__ void store8(bf16* p, const float (&f)[8]) { act::st8(p, f); }

// =============================================================================================== view attention
// reference model/Attention.py:20-23 on the stack of model/models.py:163-166, + the residual of :168-169.
//   hidden [2][M][D] = tanh(W1 z + b1) (GEMM epilogue), z [2][M][D], X [M][D]
//   w_v = w2 . hidden_v ; beta = softmax_v(w) ; embed = sum_v beta_v z_v ; Xnew = X + embed
// one warp per node row.
__global__ void __launch_bounds__(256)
view_attn_fwd_kernel(const bf16* __restrict__ hidden, const bf16* __restrict__ z, const bf16* __restrict__ X,
                     const float* __restrict__ w2, long long M, int D, bf16* __restrict__ Xnew,
                     bf16* __restrict__ embed, float* __restrict__ beta) {
  pdl_trigger();
  {   // blockIdx.y = input stream (appearance / motion): every operand of stream s follows that of stream s-1
    const long long sy = blockIdx.y;
    hidden += sy * 2 * M * D; z += sy * 2 * M * D; X += sy * M * D; w2 += sy * D; Xnew += sy * M * D; beta += sy * M * 2;
    if (embed != nullptr) embed += sy * M * D;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < M; r += (long long)gridDim.x * 8) {
    float w0 = 0.f, w1 = 0.f;
    for (int c = lane * 8; c < D; c += 256) {
      float h0[8], h1[8];
      load8(hidden + r * D + c, h0);
      load8(hidden + (M + r) * D + c, h1);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float w = w2[c + q];
        w0 += w * h0[q];
        w1 += w * h1[q];
      }
    }
    w0 = warp_sum(w0);
    w1 = warp_sum(w1);
    const float m = fmaxf(w0, w1);
    const float e0 = __expf(w0 - m), e1 = __expf(w1 - m);
    const float b0 = e0 / (e0 + e1), b1 = e1 / (e0 + e1);
    if (lane == 0) {
      beta[r * 2] = b0;
      beta[r * 2 + 1] = b1;
    }
    for (int c = lane * 8; c < D; c += 256) {
      float z0[8], z1[8], x[8], e[8];
      load8(z + r * D + c, z0);
      load8(z + (M + r) * D + c, z1);
      load8(X + r * D + c, x);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        e[q] = b0 * z0[q] + b1 * z1[q];
        x[q] += e[q];
      }
      store8(Xnew + r * D + c, x);
      if (embed != nullptr) store8(embed + r * D + c, e);
    }
  }
}

// dXnew [M][D] (+ optional dembed_ext) -> dz [2][M][D], dhid_pre [2][M][D] (tanh' applied), dw2 partial [gridDim][D]
__global__ void __launch_bounds__(256)
view_attn_bwd_kernel(const bf16* __restrict__ dXnew, const bf16* __restrict__ dembed_ext, const bf16* __restrict__ hidden,
                     const bf16* __restrict__ z, const float* __restrict__ w2, const float* __restrict__ beta,
                     long long M, int D, bf16* __restrict__ dz, bf16* __restrict__ dhid, float* __restrict__ dw2_part) {
  pdl_trigger();
  {   // blockIdx.y = input stream
    const long long sy = blockIdx.y;
    dXnew += sy * M * D; hidden += sy * 2 * M * D; z += sy * 2 * M * D; w2 += sy * D; beta += sy * M * 2;
    dz += sy * 2 * M * D; dhid += sy * 2 * M * D; dw2_part += sy * (long long)gridDim.x * D;
    if (dembed_ext != nullptr) dembed_ext += sy * M * D;
  }
  extern __shared__ float dw2_s[];   // [D]
  for (int c = threadIdx.x; c < D; c += blockDim.x) dw2_s[c] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // a lane owns the same columns (lane * 8 + 256 k) of every row it visits: dw2 accumulates in registers and reaches shared
  // memory ONCE per thread (one shared atomic per element per row was the top stall of this kernel)
  constexpr int kMaxPieces = 4;          // D <= 1024 on the register path
  float dwacc[kMaxPieces][8];
#pragma unroll
  for (int k = 0; k < kMaxPieces; ++k)
#pragma unroll
    for (int q = 0; q < 8; ++q) dwacc[k][q] = 0.f;
  const bool reg_path = D <= 256 * kMaxPieces;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < M; r += (long long)gridDim.x * 8) {
    const float b0 = beta[r * 2], b1 = beta[r * 2 + 1];
    float db0 = 0.f, db1 = 0.f;
    for (int c = lane * 8; c < D; c += 256) {
      float de[8], z0[8], z1[8], o0[8], o1[8];
      load8(dXnew + r * D + c, de);
      if (dembed_ext != nullptr) {
        float ex[8];
        load8(dembed_ext + r * D + c, ex);
#pragma unroll
        for (int q = 0; q < 8; ++q) de[q] += ex[q];
      }
      load8(z + r * D + c, z0);
      load8(z + (M + r) * D + c, z1);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        db0 += de[q] * z0[q];
        db1 += de[q] * z1[q];
        o0[q] = b0 * de[q];
        o1[q] = b1 * de[q];
      }
      store8(dz + r * D + c, o0);
      store8(dz + (M + r) * D + c, o1);
    }
    db0 = warp_sum(db0);
    db1 = warp_sum(db1);
    const float t = b0 * db0 + b1 * db1;
    const float dw0 = b0 * (db0 - t), dw1 = b1 * (db1 - t);
#pragma unroll
    for (int k = 0; k < kMaxPieces; ++k) {
      const int c = lane * 8 + 256 * k;
      if (c < D && reg_path) {
        float h0[8], h1[8], o0[8], o1[8];
        load8(hidden + r * D + c, h0);
        load8(hidden + (M + r) * D + c, h1);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float w = w2[c + q];
          o0[q] = dw0 * w * (1.f - h0[q] * h0[q]);
          o1[q] = dw1 * w * (1.f - h1[q] * h1[q]);
          dwacc[k][q] += dw0 * h0[q] + dw1 * h1[q];
        }
        store8(dhid + r * D + c, o0);
        store8(dhid + (M + r) * D + c, o1);
      }
    }
    if (!reg_path)
      for (int c = lane * 8; c < D; c += 256) {
        float h0[8], h1[8], o0[8], o1[8];
        load8(hidden + r * D + c, h0);
        load8(hidden + (M + r) * D + c, h1);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float w = w2[c + q];
          o0[q] = dw0 * w * (1.f - h0[q] * h0[q]);
          o1[q] = dw1 * w * (1.f - h1[q] * h1[q]);
          atomicAdd(&dw2_s[c + q], dw0 * h0[q] + dw1 * h1[q]);
        }
        store8(dhid + r * D + c, o0);
        store8(dhid + (M + r) * D + c, o1);
      }
  }
  if (reg_path) {
#pragma unroll
    for (int k = 0; k < kMaxPieces; ++k) {
      const int c = lane * 8 + 256 * k;
      if (c < D) {
#pragma unroll
        for (int q = 0; q < 8; ++q) atomicAdd(&dw2_s[c + q], dwacc[k][q]);
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += blockDim.x) dw2_part[(long long)blockIdx.x * D + c] = dw2_s[c];
}

// =============================================================================================== MFB pair-sum
// reference model/fusions/fusions.py:433-441: z = (x0 * x1).view(..., 256, 2).sum(-1)   (x0, x1 already ELU'd by the GEMM)
__global__ void mfb_fwd_kernel(const bf16* __restrict__ x0, const bf16* __restrict__ x1, bf16* __restrict__ z,
                               long long n_out4) {   // n_out4 = M*mm/4 ; each thread: 8 inputs -> 4 outputs
  pdl_trigger();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_out4; i += (long long)gridDim.x * blockDim.x) {
    float a[8], b[8];
    load8(x0 + i * 8, a);
    load8(x1 + i * 8, b);
    act::st2(z + i * 4, a[0] * b[0] + a[1] * b[1], a[2] * b[2] + a[3] * b[3]);
    act::st2(z + i * 4 + 2, a[4] * b[4] + a[5] * b[5], a[6] * b[6] + a[7] * b[7]);
  }
}
// dz -> dpre0 = dz_pair * x1 * ELU'(x0), dpre1 = dz_pair * x0 * ELU'(x1)
__global__ void mfb_bwd_kernel(const bf16* __restrict__ dz, const bf16* __restrict__ x0, const bf16* __restrict__ x1,
                               bf16* __restrict__ d0, bf16* __restrict__ d1, long long n_out4) {
  pdl_trigger();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_out4; i += (long long)gridDim.x * blockDim.x) {
    float a[8], b[8], oa[8], ob[8];
    load8(x0 + i * 8, a);
    load8(x1 + i * 8, b);
    const float2 d01 = act::ld2(dz + i * 4), d23 = act::ld2(dz + i * 4 + 2);
    const float d[4] = {d01.x, d01.y, d23.x, d23.y};
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      oa[q] = d[q >> 1] * b[q] * elu_grad_from_out(a[q]);
      ob[q] = d[q >> 1] * a[q] * elu_grad_from_out(b[q]);
    }
    store8(d0 + i * 8, oa);
    store8(d1 + i * 8, ob);
  }
}

// =============================================================================================== read-out
// reference model/AnswerDecoder.py:176-180: alpha = softmax_n(w . u_n + c), pooled = sum_n alpha_n v_n
//   u = ELU(v W_v^T) comes from the GEMM; v is the (already dropped-out) feature block.
__global__ void __launch_bounds__(256)
readout_fwd_kernel(const bf16* __restrict__ v, const bf16* __restrict__ u, const float* __restrict__ w,
                   const float* __restrict__ c, int N, int D, float* __restrict__ alpha, bf16* __restrict__ pooled,
                   long long ld_p) {
  pdl_trigger();
  __shared__ float sc[64];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int n = warp; n < N; n += 8) {
    float acc = 0.f;
    const bf16* row = u + ((long long)b * N + n) * D;
    for (int k = lane * 8; k < D; k += 256) {
      float f[8];
      load8(row + k, f);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc += f[q] * w[k + q];
    }
    acc = warp_sum(acc);
    if (lane == 0) sc[n] = acc + c[0];
  }
  __syncthreads();
  if (warp == 0) {
    float m = -INFINITY;
    for (int n = lane; n < N; n += 32) m = fmaxf(m, sc[n]);
    m = warp_max(m);
    float s = 0.f;
    for (int n = lane; n < N; n += 32) s += __expf(sc[n] - m);
    s = warp_sum(s);
    for (int n = lane; n < N; n += 32) {
      const float a = __expf(sc[n] - m) / s;
      sc[n] = a;
      alpha[(long long)b * N + n] = a;
    }
  }
  __syncthreads();
  for (int k = threadIdx.x * 2; k < D; k += 512) {
    float ax = 0.f, ay = 0.f;
    for (int n = 0; n < N; ++n) {
      const float2 x = act::ld2(v + ((long long)b * N + n) * D + k);
      ax += sc[n] * x.x;
      ay += sc[n] * x.y;
    }
    act::st2(pooled + (long long)b * ld_p + k, ax, ay);
  }
}

// dpooled [B][ld_p] -> dv [B][N][D] = alpha_n dpooled ; du_pre = dscore_n * w * ELU'(u) ; dw partial [B][D], dc partial [B]
__global__ void __launch_bounds__(256)
readout_bwd_kernel(const bf16* __restrict__ dpooled, long long ld_p, const bf16* __restrict__ v,
                   const bf16* __restrict__ u, const float* __restrict__ w, const float* __restrict__ alpha, int N,
                   int D, bf16* __restrict__ dv, bf16* __restrict__ du, float* __restrict__ dw_part,
                   float* __restrict__ dc_part) {
  pdl_trigger();
  __shared__ float da[64];
  __shared__ float al[64];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bf16* dp = dpooled + (long long)b * ld_p;
  for (int n = warp; n < N; n += 8) {
    float acc = 0.f;
    const bf16* row = v + ((long long)b * N + n) * D;
    for (int k = lane * 8; k < D; k += 256) {
      float f[8], g[8];
      load8(row + k, f);
      load8(dp + k, g);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc += f[q] * g[q];
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      da[n] = acc;
      al[n] = alpha[(long long)b * N + n];
    }
  }
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
    for (int n = lane; n < N; n += 32) t += al[n] * da[n];
    t = warp_sum(t);
    float dcs = 0.f;
    for (int n = lane; n < N; n += 32) {
      const float ds = al[n] * (da[n] - t);
      da[n] = ds;
      dcs += ds;
    }
    dcs = warp_sum(dcs);
    if (lane == 0) dc_part[b] = dcs;
  }
  __syncthreads();
  for (int k = threadIdx.x * 2; k < D; k += 512) {
    const float2 g = act::ld2(dp + k);
    const float w0 = w[k], w1 = w[k + 1];
    float dwx = 0.f, dwy = 0.f;
    for (int n = 0; n < N; ++n) {
      const long long off = ((long long)b * N + n) * D + k;
      act::st2(dv + off, al[n] * g.x, al[n] * g.y);
      const float2 uu = act::ld2(u + off);
      dwx += da[n] * uu.x;
      dwy += da[n] * uu.y;
      act::st2(du + off, da[n] * w0 * elu_grad_from_out(uu.x), da[n] * w1 * elu_grad_from_out(uu.y));
    }
    dw_part[(long long)b * D + k] = dwx;
    dw_part[(long long)b * D + k + 1] = dwy;
  }
}

// =============================================================================================== BatchNorm1d
// reference model/AnswerDecoder.py:193 (nn.BatchNorm1d(module_dim)): batch statistics (biased variance) in training,
// running statistics in eval; running stats updated with momentum 0.1 and the UNBIASED variance, as torch does.
// Block = 32 feature columns x kBnRL row lanes: the batch dimension is walked by kBnRL threads per column and reduced through
// shared memory in a fixed order (one thread per column walking all B rows took 100 us for the backward at B = 256; 8 row
// lanes 31 us: 24 CTAs of serial 32-row walks; 32 row lanes put 4x more loads in flight).
constexpr int kBnRL = 32;
__device__ __forceinline__ float bn_reduce8(float v, float (*red)[33], int cl, int rl) {
  __syncthreads();
  red[rl][cl] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < kBnRL; ++k) s += red[k][cl];
  return s;
}

template <typename TX>
__global__ void __launch_bounds__(32 * kBnRL)
bn_fwd_kernel(const TX* __restrict__ x, int B, int D, const float* __restrict__ gamma, const float* __restrict__ betap,
              float* __restrict__ run_mean, float* __restrict__ run_var, int training, float momentum, float eps,
              bf16* __restrict__ y, float* __restrict__ mean_out, float* __restrict__ rstd_out,
              const float* __restrict__ ext_stats, int Btot) {
  __shared__ float red[kBnRL][33];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const bool ok = c < D;
  float mean = 0.f, var = 1.f;
  if (training && ext_stats != nullptr) {
    // synchronised BatchNorm: (sum, sum of squares) over the GLOBAL batch of Btot rows, all-reduced by the caller
    if (ok) {
      mean = ext_stats[c] / Btot;
      var = fmaxf(ext_stats[D + c] / Btot - mean * mean, 0.f);
      if (rl == 0 && run_mean != nullptr) {
        run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * mean;
        run_var[c] = (1.f - momentum) * run_var[c] + momentum * (Btot > 1 ? var * Btot / (Btot - 1) : var);
      }
    }
  } else if (training) {
    float s = 0.f;
    if (ok)
      for (int r = rl; r < B; r += kBnRL) s += ldf<TX>(x + (long long)r * D + c);
    mean = bn_reduce8(s, red, cl, rl) / B;
    float v = 0.f;
    if (ok)
      for (int r = rl; r < B; r += kBnRL) {
        const float d = ldf<TX>(x + (long long)r * D + c) - mean;
        v += d * d;
      }
    v = bn_reduce8(v, red, cl, rl);
    var = v / B;
    if (ok && rl == 0 && run_mean != nullptr) {
      run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * mean;
      run_var[c] = (1.f - momentum) * run_var[c] + momentum * (B > 1 ? v / (B - 1) : var);
    }
  } else if (ok) {
    mean = run_mean[c];
    var = run_var[c];
  }
  if (!ok) return;
  const float rstd = rsqrtf(var + eps);
  if (rl == 0 && mean_out != nullptr) {
    mean_out[c] = mean;
    rstd_out[c] = rstd;
  }
  const float g = gamma[c], bt = betap[c];
  for (int r = rl; r < B; r += kBnRL)
    act::st1(y + (long long)r * D + c, (ldf<TX>(x + (long long)r * D + c) - mean) * rstd * g + bt);
}

// per-column (sum, sum of squares) of the local batch: out [2][D] (the operand of the SyncBN all-reduce)
template <typename TX>
__global__ void __launch_bounds__(32 * kBnRL) bn_stats_kernel(const TX* __restrict__ x, int B, int D, float* __restrict__ out) {
  __shared__ float red[kBnRL][33];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const bool ok = c < D;
  float s = 0.f, ss = 0.f;
  if (ok)
    for (int r = rl; r < B; r += kBnRL) {
      const float v = ldf<TX>(x + (long long)r * D + c);
      s += v;
      ss += v * v;
    }
  s = bn_reduce8(s, red, cl, rl);
  ss = bn_reduce8(ss, red, cl, rl);
  if (ok && rl == 0) {
    out[c] = s;
    out[D + c] = ss;
  }
}

// ext_sums [2][D] = (sum dy, sum dy * xhat) over the GLOBAL batch of Btot rows (SyncBN, second pass); stats_only: write the
// LOCAL sums to dbeta / dgamma and stop (SyncBN, first pass)
template <typename TX>
__global__ void __launch_bounds__(32 * kBnRL)
bn_bwd_kernel(const bf16* __restrict__ dy, const TX* __restrict__ x, int B, int D, const float* __restrict__ gamma,
              const float* __restrict__ mean, const float* __restrict__ rstd, int training, TX* __restrict__ dx,
              float* __restrict__ dgamma, float* __restrict__ dbeta, const float* __restrict__ ext_sums, int Btot,
              int stats_only) {
  __shared__ float red[kBnRL][33];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const bool ok = c < D;
  const float m = ok ? mean[c] : 0.f, rs = ok ? rstd[c] : 0.f, g = ok ? gamma[c] : 0.f;
  float sdy = 0.f, sdyx = 0.f;
  if (ok)
    for (int r = rl; r < B; r += kBnRL) {
      const float d = act::ld1(dy + (long long)r * D + c);
      const float xh = (ldf<TX>(x + (long long)r * D + c) - m) * rs;
      sdy += d;
      sdyx += d * xh;
    }
  sdy = bn_reduce8(sdy, red, cl, rl);
  sdyx = bn_reduce8(sdyx, red, cl, rl);
  if (!ok) return;
  if (rl == 0 && dgamma != nullptr) {
    dgamma[c] = sdyx;
    dbeta[c] = sdy;
  }
  if (stats_only) return;
  float nb = (float)B;
  if (ext_sums != nullptr) {
    sdy = ext_sums[c];
    sdyx = ext_sums[D + c];
    nb = (float)Btot;
  }
  for (int r = rl; r < B; r += kBnRL) {
    const float d = act::ld1(dy + (long long)r * D + c);
    const float xh = (ldf<TX>(x + (long long)r * D + c) - m) * rs;
    const float o = training ? g * rs * (d - sdy / nb - xh * sdyx / nb) : g * rs * d;
    stf<TX>(dx + (long long)r * D + c, o);
  }
}

// =============================================================================================== cross-entropy
// nn.CrossEntropyLoss (mean) at train.py:121,146: loss_part[b] = -log softmax(logits_b)[ans_b] / B,
// dlogits = (softmax - onehot) * scale / B  (bf16, row stride ld_d, padding columns zeroed)
template <typename TG>
__global__ void ce_kernel(const float* __restrict__ logits, const long long* __restrict__ ans, int B, int A,
                          float scale, float* __restrict__ loss_part, TG* __restrict__ dlogits, long long ld_d,
                          int* __restrict__ correct) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= B) return;
  const float* row = logits + (long long)b * A;
  float m = -INFINITY;
  int am = 0;
  for (int a = lane; a < A; a += 32) {
    if (row[a] > m) { m = row[a]; am = a; }
  }
  // warp arg-max (first index wins on ties, like torch.argmax / batch_accuracy at train.py:352-356)
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, o);
    const int oa = __shfl_xor_sync(0xffffffffu, am, o);
    if (om > m || (om == m && oa < am)) { m = om; am = oa; }
  }
  float s = 0.f;
  for (int a = lane; a < A; a += 32) s += __expf(row[a] - m);
  s = warp_sum(s);
  const long long t = ans[b];
  const float lse = m + __logf(s);
  if (lane == 0) {
    loss_part[b] = (lse - row[t]) / B;
    if (correct != nullptr) correct[b] = (am == (int)t) ? 1 : 0;
  }
  if (dlogits != nullptr) {
    for (int a = lane; a < ld_d; a += 32) {
      float g = 0.f;
      if (a < A) g = (__expf(row[a] - lse) - (a == t ? 1.f : 0.f)) * scale / B;
      stf<TG>(dlogits + (long long)b * ld_d + a, g);
    }
  }
}


// =============================================================================================== validation counters
// reference validate.py:59-134: preds = argmax(logits), agreeings = preds == answers, then per-question-type bookkeeping in
// Python loops over the batch (a host sync per sample: int(category.cpu()), vocab look-ups per key word). Here: one warp per
// sample — argmax (first index wins on ties, like torch.argmax), category from the SVQA category id or from the question's
// first token through a [V] token->type table, and two atomic counters per category: counts[cat] = {correct, total}; row
// n_cat holds the totals over all samples (uncategorised samples only count there).
__global__ void accuracy_counters_kernel(const float* __restrict__ logits, const long long* __restrict__ answers, int B, int A,
                                         const long long* __restrict__ category, const long long* __restrict__ tokens,
                                         long long ld_tok, const int* __restrict__ token_to_cat, int V, int n_cat,
                                         long long* __restrict__ counts, int* __restrict__ preds) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= B) return;
  const float* row = logits + (long long)b * A;
  float m = -INFINITY;
  int am = 0;
  for (int a = lane; a < A; a += 32)
    if (row[a] > m) { m = row[a]; am = a; }
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, o);
    const int oa = __shfl_xor_sync(0xffffffffu, am, o);
    if (om > m || (om == m && oa < am)) { m = om; am = oa; }
  }
  if (lane != 0) return;
  if (preds != nullptr) preds[b] = am;
  const unsigned long long ok = (am == (int)answers[b]) ? 1ull : 0ull;
  int cat = -1;
  if (category != nullptr) {
    cat = (int)category[b];
  } else if (tokens != nullptr && token_to_cat != nullptr) {
    const long long tok = tokens[(long long)b * ld_tok];
    if (tok >= 0 && tok < V) cat = token_to_cat[tok];
  }
  unsigned long long* c = reinterpret_cast<unsigned long long*>(counts);
  if (cat >= 0 && cat < n_cat) {
    atomicAdd(c + 2 * cat, ok);
    atomicAdd(c + 2 * cat + 1, 1ull);
  }
  atomicAdd(c + 2 * n_cat, ok);
  atomicAdd(c + 2 * n_cat + 1, 1ull);
}

// =============================================================================================== streaming helpers
// Appearance prologue, reference model/Preprocessing.py:220-223: tanh(dropout(x)) and the [B,N,F,C] -> [F, B*N, C]
// re-layout (two full transposed copies in the reference) fused with the fp32 -> bf16 cast in ONE pass.
// TIN = float (the reference's feature format) or bf16 (features stored / shipped as bf16: half the host-to-device bytes)
template <typename TIN>
__device__ __forceinline__ void prep_item(const TIN* __restrict__ in, bf16* __restrict__ out, long long i, float (&f)[8],
                                          long long S, int T, int c8, int do_tanh, int time_major, const DropoutCfg& dc) {
  if (dc.p > 0.f) {
    float sc[8];
    dropout_scale8(dc, i, sc);
#pragma unroll
    for (int q = 0; q < 8; ++q) f[q] *= sc[q];
  }
  if (do_tanh) {
#pragma unroll
    for (int q = 0; q < 8; ++q) f[q] = tanh_fast(f[q]);   // output is bf16: the 2^-11 approximation is below its ulp
  }
  long long o = i;
  if (time_major) {
    // (32-bit index arithmetic whenever the tensor allows it: two 64-bit divisions per item were a third of the kernel's
    //  instructions)
    if (i < 0x7fffffffLL) {
      const unsigned iu = (unsigned)i, row = iu / (unsigned)c8, cc = iu - row * (unsigned)c8;
      const unsigned s_ = row / (unsigned)T, t = row - s_ * (unsigned)T;
      o = ((long long)t * S + s_) * c8 + cc;
    } else {
      const long long row = i / c8;     // = s * T + t
      const int cc = (int)(i - row * c8);
      const long long s_ = row / T;
      const int t = (int)(row - s_ * T);
      o = ((long long)t * S + s_) * c8 + cc;
    }
  }
  store8(out + o * 8, f);
}

// Gathered input (GATHER): `in` is a feature store [V][N][T][C] resident in device memory and batch item b is video
// rows[b]; everything else (item index i, output layout, dropout mask keyed by i) is that of the dense pass over the
// batch store[rows]. The batch side keeps 32-bit index arithmetic; the store offset rows[b]*N*T*C is 64-bit (a store
// passes 2^31 elements at ~3300 SVQA videos). A row outside [0, V) is never read: its items are zeros (tanh(0) = 0, so its
// output rows are zero) and the sticky word *err is set.
struct GatherCfg {
  const int* rows;
  long long V;
  int slab8;      // N * T * C / 8: 8-element items per video
  int* err;
};

template <typename TIN, bool GATHER>
__device__ __forceinline__ void prep_load(const TIN* __restrict__ in, long long i, float (&f)[8], const GatherCfg& g) {
  if constexpr (!GATHER) {
    load8g(in + i * 8, f);
  } else {
    long long b, w;
    if (i < 0x7fffffffLL) {
      const unsigned iu = (unsigned)i, bu = iu / (unsigned)g.slab8;
      b = bu;
      w = iu - bu * (unsigned)g.slab8;
    } else {
      b = i / g.slab8;
      w = i - b * g.slab8;
    }
    const int r = __ldg(g.rows + b);
    if (r < 0 || r >= g.V) {
#pragma unroll
      for (int q = 0; q < 8; ++q) f[q] = 0.f;
      *g.err = 1;
      return;
    }
    load8g(in + ((long long)r * g.slab8 + w) * 8, f);
  }
}

template <typename TIN, bool GATHER>
__global__ void prep_features_kernel(const TIN* __restrict__ in, bf16* __restrict__ out, long long S, int T, int C,
                                     int do_tanh, int time_major, DropoutCfg dc, GatherCfg g) {
  const long long n8 = S * T * (long long)C / 8;
  const int c8 = C / 8;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  for (; i + stride < n8; i += 2 * stride) {      // two items per trip: both loads are in flight before either is consumed
    float f0[8], f1[8];
    prep_load<TIN, GATHER>(in, i, f0, g);
    prep_load<TIN, GATHER>(in, i + stride, f1, g);
    prep_item<TIN>(in, out, i, f0, S, T, c8, do_tanh, time_major, dc);
    prep_item<TIN>(in, out, i + stride, f1, S, T, c8, do_tanh, time_major, dc);
  }
  if (i < n8) {
    float f0[8];
    prep_load<TIN, GATHER>(in, i, f0, g);
    prep_item<TIN>(in, out, i, f0, S, T, c8, do_tanh, time_major, dc);
  }
}

// fp32 [rows][cols] (ld_in) -> bf16 [rows][out_cols] (ld_out), zero padded columns; optional LSTM gate interleave:
// output row 4*j + g <- input row g*H + j  (nn.LSTM stores i|f|g|o blocks; the fused cell wants them per unit).
__global__ void cast_rows_kernel(const float* __restrict__ in, long long ld_in, bf16* __restrict__ out, long long ld_out,
                                 int rows, int cols, int out_cols, int lstm_H) {
  pdl_trigger();
  const long long total = (long long)rows * out_cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / out_cols), c = (int)(i - (long long)r * out_cols);
    int src = r;
    if (lstm_H > 0) src = (r & 3) * lstm_H + (r >> 2);
    out[(long long)r * ld_out + c] = __float2bfloat16_rn(c < cols ? in[(long long)src * ld_in + c] : 0.f);
  }
}


// fp32 -> three bf16 planes [lo | hi | hi] ([3][rows][ld_out]): the operand format of the fp32-accurate ("3 x bf16") GEMM.
// x = hi + lo + r with |r| <= 2^-17 |x|; a product a.b is evaluated as a_lo b_hi + a_hi b_hi + a_hi b_lo by ONE tcgen05 GEMM
// whose reduction runs over the three planes: the A operand reads them in the order 0, 1, 2, the B operand in the order 2, 1, 0.
__global__ void split3_kernel(const float* __restrict__ in, long long ld_in, int rows, int cols, bf16* __restrict__ out,
                              long long ld_out, long long plane) {
  pdl_trigger();
  const int c8 = (int)(ld_out >> 3);
  const long long total = (long long)rows * c8;
  const bool vec_in = ((ld_in & 3) == 0) && ((reinterpret_cast<uintptr_t>(in) & 15) == 0);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / c8), c = (int)(i - (long long)r * c8) * 8;
    const float* row = in + (long long)r * ld_in + c;
    float f[8], hi[8], lo[8];
    if (vec_in && c + 8 <= cols) {
      load8g(row, f);
    } else {
#pragma unroll
      for (int q = 0; q < 8; ++q) f[q] = (c + q < cols) ? row[q] : 0.f;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      hi[q] = __bfloat162float(__float2bfloat16_rn(f[q]));
      lo[q] = f[q] - hi[q];
    }
    bf16* o = out + (long long)r * ld_out + c;
    store8(o, lo);
    store8(o + plane, hi);
    store8(o + 2 * plane, hi);
  }
}

// out = in * dropout mask (the same kernel is its own backward)
__global__ void dropout_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, long long n8, DropoutCfg dc) {
  pdl_trigger();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float f[8], sc[8];
    load8(in + i * 8, f);
    dropout_scale8(dc, i, sc);
#pragma unroll
    for (int q = 0; q < 8; ++q) f[q] *= sc[q];
    store8(out + i * 8, f);
  }
}

// out = dy * dropout mask * act'(y)   (y is the activation OUTPUT; act: 0 none, 1 ELU, 2 tanh); optional accumulate
__global__ void act_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ y, bf16* __restrict__ out,
                               long long n8, int act, int accumulate, DropoutCfg dc) {
  pdl_trigger();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float d[8], yy[8];
    load8(dy + i * 8, d);
    if (dc.p > 0.f) {
      float sc[8];
      dropout_scale8(dc, i, sc);
#pragma unroll
      for (int q = 0; q < 8; ++q) d[q] *= sc[q];
    }
    if (act != 0) {
      load8(y + i * 8, yy);
#pragma unroll
      for (int q = 0; q < 8; ++q) d[q] *= (act == 1) ? elu_grad_from_out(yy[q]) : (1.f - yy[q] * yy[q]);
    }
    if (accumulate) {
      float o[8];
      load8(out + i * 8, o);
#pragma unroll
      for (int q = 0; q < 8; ++q) d[q] += o[q];
    }
    store8(out + i * 8, d);
  }
}


// Up to 4 dropped copies of (up to 4) inputs in ONE launch: the four graphs of a DualVGR unit each read their own dropped copy
// of their stream (reference model/GraphNN.py:175, one F.dropout per punishGAT call). blockIdx.y = copy.
struct DropMulti {
  const bf16* in[4];
  bf16* out[4];
  unsigned int stream[4];
};
__global__ void dropout_multi_kernel(const DropMulti m, long long n8, DropoutCfg dc) {
  pdl_trigger();
  const int y = blockIdx.y;
  dc.stream = m.stream[y];
  const bf16* __restrict__ in = m.in[y];
  bf16* __restrict__ out = m.out[y];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float f[8], sc[8];
    load8(in + i * 8, f);
    dropout_scale8(dc, i, sc);
#pragma unroll
    for (int q = 0; q < 8; ++q) f[q] *= sc[q];
    store8(out + i * 8, f);
  }
}

// Backward of those copies, summed per stream and merged with the gradient that bypasses the graphs (the residual branch):
//   dX[s] = base[s] + sum_{g in stream s} mask_g * dxt[g]          blockIdx.y = stream
struct GatInBwd {
  const bf16* dxt[4];
  unsigned int stream[4];
  const bf16* base[2];
  bf16* out[2];
  int per_stream;
};
__global__ void gat_input_bwd_kernel(const GatInBwd m, long long n8, DropoutCfg dc) {
  pdl_trigger();
  const int s = blockIdx.y;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float acc[8];
    if (m.base[s] != nullptr) {
      load8(m.base[s] + i * 8, acc);
    } else {
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] = 0.f;
    }
    for (int j = 0; j < m.per_stream; ++j) {
      const int g = s * m.per_stream + j;
      float d[8], sc[8];
      load8(m.dxt[g] + i * 8, d);
      dc.stream = m.stream[g];
      dropout_scale8(dc, i, sc);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] += d[q] * sc[q];
    }
    store8(m.out[s] + i * 8, acc);
  }
}

// Question-word prologue, reference model/Preprocessing.py:109-111: words = tanh(dropout(embedding[tokens])) written twice
// in one pass — [B][L][Wp] (operand of QueryAttn) and time-major [L][B][Wp] (TMA operand of the question LSTMs) — both bf16
// with the word dimension zero-padded to Wp (16-byte rows). Replaces the embedding gather, dropout, tanh, pad, transpose and
// cast launches of the eager path.
__global__ void embed_fwd_kernel(const long long* __restrict__ tokens, const float* __restrict__ table, int B, int L, int W,
                                 int Wp, bf16* __restrict__ words, bf16* __restrict__ x_tm, DropoutCfg dc) {
  pdl_trigger();
  const int w8 = Wp / 8;
  const long long n8 = (long long)B * L * w8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / w8;       // = b * L + l
    const int c0 = (int)(i - row * w8) * 8;
    const long long tok = tokens[row];
    float f[8], sc[8];
    dropout_scale8(dc, i, sc);
#pragma unroll
    for (int q = 0; q < 8; ++q) f[q] = (c0 + q < W) ? tanhf_(table[tok * W + c0 + q] * sc[q]) : 0.f;
    store8(words + i * 8, f);
    const long long b = row / L;
    const int l = (int)(row - b * L);
    store8(x_tm + (((long long)l * B + b) * Wp + c0), f);
  }
}
// dtable[tok] += (d_words[b][l] + d_x[l][b]) * tanh'(words) * mask   (fp32 atomics: tokens repeat across the batch)
__global__ void embed_bwd_kernel(const long long* __restrict__ tokens, const bf16* __restrict__ words,
                                 const bf16* __restrict__ d_words, const bf16* __restrict__ d_x_tm, int B, int L, int W, int Wp,
                                 float* __restrict__ dtable, DropoutCfg dc) {
  pdl_trigger();
  const int w8 = Wp / 8;
  const long long n8 = (long long)B * L * w8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / w8;
    const int c0 = (int)(i - row * w8) * 8;
    const long long tok = tokens[row];
    const long long b = row / L;
    const int l = (int)(row - b * L);
    float w[8], d[8], sc[8];
    load8(words + i * 8, w);
#pragma unroll
    for (int q = 0; q < 8; ++q) d[q] = 0.f;
    if (d_words != nullptr) load8(d_words + i * 8, d);
    if (d_x_tm != nullptr) {
      float e[8];
      load8(d_x_tm + (((long long)l * B + b) * Wp + c0), e);
#pragma unroll
      for (int q = 0; q < 8; ++q) d[q] += e[q];
    }
    dropout_scale8(dc, i, sc);
    float g[8];
    bool any = false;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      g[q] = (c0 + q < W) ? d[q] * (1.f - w[q] * w[q]) * sc[q] : 0.f;
      any |= g[q] != 0.f;
    }
    if (!any) continue;                      // padded positions / dropped octets: nothing to add
    float* dst = dtable + tok * W + c0;
    if ((W & 3) == 0 && c0 + 8 <= W && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      // two 16-byte vector reductions instead of eight scalar atomics (the scalar version was atomic-throughput bound)
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(g[0]), "f"(g[1]), "f"(g[2]), "f"(g[3]) : "memory");
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4), "f"(g[4]), "f"(g[5]), "f"(g[6]), "f"(g[7]) : "memory");
    } else {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (c0 + q < W && g[q] != 0.f) atomicAdd(dst + q, g[q]);
    }
  }
}

// ---- LSTM operand packing (one launch each instead of a chain of tiny framework kernels per train step)
// Several cast_rows problems in one launch (blockIdx.y = problem): the bf16 gate-interleaved copies of all W_ih / W_hh matrices
// of an encoder (2 - 4 directions) written into ONE row-concatenated operand.
constexpr int kMaxCast = 8;
struct CastGroup {
  const float* in[kMaxCast];
  bf16* out[kMaxCast];
  long long ld_in[kMaxCast];
  int rows[kMaxCast], cols[kMaxCast];
  long long ld_out;
  int out_cols, lstm_H;
};
__global__ void cast_rows_grouped_kernel(const CastGroup G) {
  pdl_trigger();
  const int y = blockIdx.y;
  const float* __restrict__ in = G.in[y];
  bf16* __restrict__ out = G.out[y];
  const int cols = G.cols[y];
  const long long ld_in = G.ld_in[y];
  if ((G.out_cols & 7) == 0 && (G.ld_out & 7) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    // 8 columns per thread: two 16-byte loads (when the source row allows it), one 16-byte store
    const int oc8 = G.out_cols >> 3;
    const bool vec_in = ((ld_in & 3) == 0) && ((reinterpret_cast<uintptr_t>(in) & 15) == 0);
    const long long total = (long long)G.rows[y] * oc8;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const int r = (int)(i / oc8), c = (int)(i - (long long)r * oc8) * 8;
      int src = r;
      if (G.lstm_H > 0) src = (r & 3) * G.lstm_H + (r >> 2);
      const float* row = in + (long long)src * ld_in + c;
      float f[8];
      if (vec_in && c + 8 <= cols) {
        load8g(row, f);
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) f[q] = (c + q < cols) ? row[q] : 0.f;
      }
      store8(out + (long long)r * G.ld_out + c, f);
    }
    return;
  }
  const long long total = (long long)G.rows[y] * G.out_cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / G.out_cols), c = (int)(i - (long long)r * G.out_cols);
    int src = r;
    if (G.lstm_H > 0) src = (r & 3) * G.lstm_H + (r >> 2);
    out[(long long)r * G.ld_out + c] = __float2bfloat16_rn(c < cols ? in[(long long)src * ld_in + c] : 0.f);
  }
}
// bias[d][4j + g] = b_ih[d][g*H + j] + b_hh[d][g*H + j]   (the fused cell's gate-interleaved bias, all directions at once)
struct BiasGroup {
  const float* b_ih[4];
  const float* b_hh[4];
};
__global__ void lstm_pack_bias_kernel(const BiasGroup G, int H, float* __restrict__ out) {
  pdl_trigger();
  const int d = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * H; i += gridDim.x * blockDim.x) {
    const int src = (i & 3) * H + (i >> 2);
    out[(long long)d * 4 * H + i] = G.b_ih[d][src] + G.b_hh[d][src];
  }
}
// Gradients arriving at the question encoder (model/Preprocessing.py:112-123) packed for dvgr_lstm_seq_bwd in one pass:
//   d_seq [B][L][ld_seq] bf16 (per-token states of directions 0 .. nd_seq-1, H columns each; may be null)
//     -> dh_seq blocked [T][D][RB][H/8][32][8] (zeros for the other directions and the padded rows)
//   d_last [B][ld_last] bf16 (final states of directions d_last0 .. D-1; may be null) -> dh_last [B][D*H] (zeros elsewhere)
__global__ void lstm_pack_dh_kernel(const bf16* __restrict__ d_seq, long long ld_seq, int nd_seq, const bf16* __restrict__ d_last,
                                    long long ld_last, int d_last0, int S, int T, int D, int H, bf16* __restrict__ dh_seq,
                                    bf16* __restrict__ dh_last) {
  pdl_trigger();
  const int RB = (S + 31) / 32, UG = H / 8;
  const long long n_seq = (long long)T * D * RB * UG * 32;          // 16-byte pieces of dh_seq
  const long long n_last = (long long)S * D * UG;                   // 16-byte pieces of dh_last
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_seq + n_last; i += (long long)gridDim.x * blockDim.x) {
    uint4 v = make_uint4(0, 0, 0, 0);
    if (i < n_seq) {
      const int r = (int)(i & 31);
      long long rest = i >> 5;
      const int ug = (int)(rest % UG); rest /= UG;
      const int rb = (int)(rest % RB); rest /= RB;
      const int d = (int)(rest % D);
      const int t = (int)(rest / D);
      const int seq = rb * 32 + r;
      if (d_seq != nullptr && d < nd_seq && seq < S)
        v = *reinterpret_cast<const uint4*>(d_seq + ((long long)seq * T + t) * ld_seq + (long long)d * H + ug * 8);
      reinterpret_cast<uint4*>(dh_seq)[i] = v;
    } else {
      const long long j = i - n_seq;
      const int ug = (int)(j % UG);
      const long long rest = j / UG;
      const int d = (int)(rest % D);
      const int seq = (int)(rest / D);
      if (d_last != nullptr && d >= d_last0)
        v = *reinterpret_cast<const uint4*>(d_last + (long long)seq * ld_last + (long long)(d - d_last0) * H + ug * 8);
      reinterpret_cast<uint4*>(dh_last)[j] = v;
    }
  }
}

// a (+)= b elementwise (bf16), used to merge gradient branches
__global__ void add_kernel(bf16* __restrict__ a, const bf16* __restrict__ b, long long n8) {
  pdl_trigger();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float x[8], y[8];
    load8(a + i * 8, x);
    load8(b + i * 8, y);
#pragma unroll
    for (int q = 0; q < 8; ++q) x[q] += y[q];
    store8(a + i * 8, x);
  }
}

// Column sums, two deterministic passes: partial[chunk][C] then out[C] (+)= sum_chunk. Input bf16 or fp32.
// Block = 32 column groups (8 columns each, one 128-bit / 2x128-bit load per row) x 8 row lanes; every thread keeps
// 4 independent row loads in flight (the first version issued one dependent 2-byte load per iteration and was
// latency-bound at ~1 % of HBM bandwidth on the [81920, 3072] LSTM bias gradient).
template <typename T>
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const T* __restrict__ in, long long ld, long long R, int C, int rows_per_chunk,
                      float* __restrict__ partial, int vec_ok, long long in_batch) {
  pdl_trigger();
  __shared__ float red[8][32][9];
  in += (long long)blockIdx.z * in_batch;                        // batched call: one reduction per blockIdx.z
  partial += (long long)blockIdx.z * gridDim.y * C;
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c0 = (blockIdx.x * 32 + cg) * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_chunk;
  const long long r1 = min(R, r0 + rows_per_chunk);
  float acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.f;
  if (c0 < C) {
    if (vec_ok && c0 + 8 <= C) {
      long long r = r0 + rl;
      for (; r + 24 < r1; r += 32) {
        float f0[8], f1[8], f2[8], f3[8];
        load8g(in + r * ld + c0, f0);
        load8g(in + (r + 8) * ld + c0, f1);
        load8g(in + (r + 16) * ld + c0, f2);
        load8g(in + (r + 24) * ld + c0, f3);
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] += (f0[q] + f1[q]) + (f2[q] + f3[q]);
      }
      for (; r < r1; r += 8) {
        float f0[8];
        load8g(in + r * ld + c0, f0);
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] += f0[q];
      }
    } else {
      for (long long r = r0 + rl; r < r1; r += 8)
        for (int q = 0; q < 8; ++q)
          if (c0 + q < C) acc[q] += ldf<T>(in + r * ld + c0 + q);
    }
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) red[rl][cg][q] = acc[q];
  __syncthreads();
  if (rl == 0 && c0 < C) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += red[k][cg][q];
      if (c0 + q < C) partial[(long long)blockIdx.y * C + c0 + q] = s;
    }
  }
}
// 32 columns x 8 chunk lanes per block: the chain of dependent adds per column is chunks / 8 long instead of chunks
// (a [160 x 768] reduction took 13 us as one thread per column), summed in a fixed order -> still deterministic.
__global__ void __launch_bounds__(256)
colsum_final_kernel(const float* __restrict__ partial, int chunks, int C, float* __restrict__ out, int accumulate,
                    float scale, long long out_batch) {
  pdl_trigger();
  __shared__ float red[8][33];
  partial += (long long)blockIdx.z * chunks * C;
  out += (long long)blockIdx.z * out_batch;
  const int cl = threadIdx.x & 31, kl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  float a0 = 0.f, a1 = 0.f;
  if (c < C) {
    int k = kl;
    for (; k + 8 < chunks; k += 16) {
      a0 += partial[(long long)k * C + c];
      a1 += partial[(long long)(k + 8) * C + c];
    }
    if (k < chunks) a0 += partial[(long long)k * C + c];
  }
  red[kl][cl] = a0 + a1;
  __syncthreads();
  if (kl == 0 && c < C) {
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) acc += red[q][cl];
    acc *= scale;
    out[c] = accumulate ? out[c] + acc : acc;
  }
}

static inline int grid_for(long long n, int threads = 256, int max_blocks = 148 * 16) {
  long long b = (n + threads - 1) / threads;
  if (b < 1) b = 1;
  return (int)std::min<long long>(b, max_blocks);
}

}  // namespace DVGR_VNS
}  // namespace dvgr

using namespace dvgr;
using namespace dvgr::DVGR_VNS;
#define ST(s) reinterpret_cast<cudaStream_t>(s)
#define BF(p) reinterpret_cast<bf16*>(p)
#define CBF(p) reinterpret_cast<const bf16*>(p)

extern "C" int DVGR_FN(dvgr_view_attn_fwd_multi)(const void* hidden, const void* z, const void* x, const float* w2, long long M,
                                        int D, int n_streams, void* xnew, void* embed, float* beta, void* stream) {
  if (M <= 0 || n_streams <= 0) return 0;
  if (D % 8 != 0) return set_error("view_attn: D=%d must be a multiple of 8", D);
  view_attn_fwd_kernel<<<dim3(grid_for(M, 8, 148 * 8 / n_streams), n_streams), 256, 0, ST(stream)>>>(
      CBF(hidden), CBF(z), CBF(x), w2, M, D, BF(xnew), BF(embed), beta);
  DVGR_CHECK_LAUNCH("view_attn_fwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_view_attn_fwd)(const void* hidden, const void* z, const void* x, const float* w2, long long M, int D,
                                  void* xnew, void* embed, float* beta, void* stream) {
  return DVGR_FN(dvgr_view_attn_fwd_multi)(hidden, z, x, w2, M, D, 1, xnew, embed, beta, stream);
}

extern "C" int DVGR_FN(dvgr_view_attn_bwd_blocks)(long long M) { return grid_for(M, 8, 148 * 2); }

extern "C" int DVGR_FN(dvgr_view_attn_bwd_multi)(const void* dxnew, const void* dembed_ext, const void* hidden, const void* z,
                                        const float* w2, const float* beta, long long M, int D, int n_streams, void* dz,
                                        void* dhid, float* dw2_part, void* stream) {
  if (M <= 0 || n_streams <= 0) return 0;
  if (D % 8 != 0) return set_error("view_attn: D=%d must be a multiple of 8", D);
  const int blocks = DVGR_FN(dvgr_view_attn_bwd_blocks)(M);
  view_attn_bwd_kernel<<<dim3(blocks, n_streams), 256, D * sizeof(float), ST(stream)>>>(
      CBF(dxnew), CBF(dembed_ext), CBF(hidden), CBF(z), w2, beta, M, D, BF(dz), BF(dhid), dw2_part);
  DVGR_CHECK_LAUNCH("view_attn_bwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_view_attn_bwd)(const void* dxnew, const void* dembed_ext, const void* hidden, const void* z,
                                  const float* w2, const float* beta, long long M, int D, void* dz, void* dhid,
                                  float* dw2_part, void* stream) {
  return DVGR_FN(dvgr_view_attn_bwd_multi)(dxnew, dembed_ext, hidden, z, w2, beta, M, D, 1, dz, dhid, dw2_part, stream);
}

extern "C" int DVGR_FN(dvgr_mfb_fwd)(const void* x0, const void* x1, void* z, long long M, int mm2, void* stream) {
  if (mm2 % 8 != 0) return set_error("mfb: 2*mm_dim=%d must be a multiple of 8", mm2);
  const long long n = M * mm2 / 8;
  if (n <= 0) return 0;
  mfb_fwd_kernel<<<grid_for(n), 256, 0, ST(stream)>>>(CBF(x0), CBF(x1), BF(z), n);
  DVGR_CHECK_LAUNCH("mfb_fwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_mfb_bwd)(const void* dz, const void* x0, const void* x1, void* d0, void* d1, long long M, int mm2,
                            void* stream) {
  if (mm2 % 8 != 0) return set_error("mfb: 2*mm_dim=%d must be a multiple of 8", mm2);
  const long long n = M * mm2 / 8;
  if (n <= 0) return 0;
  mfb_bwd_kernel<<<grid_for(n), 256, 0, ST(stream)>>>(CBF(dz), CBF(x0), CBF(x1), BF(d0), BF(d1), n);
  DVGR_CHECK_LAUNCH("mfb_bwd");
  return 0;
}

extern "C" int DVGR_FN(dvgr_readout_fwd)(const void* v, const void* u, const float* w, const float* c, int B, int N, int D,
                                float* alpha, void* pooled, long long ld_p, void* stream) {
  if (B <= 0) return 0;
  if (N > 64) return set_error("readout: N=%d > 64", N);
  if (D % 8 != 0) return set_error("readout: D=%d must be a multiple of 8", D);
  readout_fwd_kernel<<<B, 256, 0, ST(stream)>>>(CBF(v), CBF(u), w, c, N, D, alpha, BF(pooled), ld_p);
  DVGR_CHECK_LAUNCH("readout_fwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_readout_bwd)(const void* dpooled, long long ld_p, const void* v, const void* u, const float* w,
                                const float* alpha, int B, int N, int D, void* dv, void* du, float* dw_part,
                                float* dc_part, void* stream) {
  if (B <= 0) return 0;
  if (N > 64) return set_error("readout: N=%d > 64", N);
  if (D % 8 != 0) return set_error("readout: D=%d must be a multiple of 8", D);
  readout_bwd_kernel<<<B, 256, 0, ST(stream)>>>(CBF(dpooled), ld_p, CBF(v), CBF(u), w, alpha, N, D, BF(dv), BF(du),
                                                dw_part, dc_part);
  DVGR_CHECK_LAUNCH("readout_bwd");
  return 0;
}

extern "C" int DVGR_FN(dvgr_bn_fwd_ex)(const void* x, int x_is_f32, int B, int D, const float* gamma, const float* beta,
                              float* run_mean, float* run_var, int training, float momentum, float eps, void* y,
                              float* mean_out, float* rstd_out, const float* ext_stats, int Btot, void* stream) {
  if (B <= 0 || D <= 0) return 0;
  if (ext_stats != nullptr && Btot < B) return set_error("bn_fwd: global batch %d smaller than the local one %d", Btot, B);
  if (x_is_f32)
    bn_fwd_kernel<float><<<(D + 31) / 32, 32 * kBnRL, 0, ST(stream)>>>(reinterpret_cast<const float*>(x), B, D, gamma, beta,
                                                                 run_mean, run_var, training, momentum, eps, BF(y),
                                                                 mean_out, rstd_out, ext_stats, Btot);
  else
    bn_fwd_kernel<bf16><<<(D + 31) / 32, 32 * kBnRL, 0, ST(stream)>>>(CBF(x), B, D, gamma, beta, run_mean, run_var, training,
                                                                momentum, eps, BF(y), mean_out, rstd_out, ext_stats, Btot);
  DVGR_CHECK_LAUNCH("bn_fwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_bn_fwd)(const void* x, int x_is_f32, int B, int D, const float* gamma, const float* beta,
                           float* run_mean, float* run_var, int training, float momentum, float eps, void* y,
                           float* mean_out, float* rstd_out, void* stream) {
  return DVGR_FN(dvgr_bn_fwd_ex)(x, x_is_f32, B, D, gamma, beta, run_mean, run_var, training, momentum, eps, y, mean_out, rstd_out,
                        nullptr, B, stream);
}
extern "C" int DVGR_FN(dvgr_bn_stats)(const void* x, int x_is_f32, int B, int D, float* out, void* stream) {
  if (B <= 0 || D <= 0) return 0;
  if (x_is_f32) bn_stats_kernel<float><<<(D + 31) / 32, 32 * kBnRL, 0, ST(stream)>>>(reinterpret_cast<const float*>(x), B, D, out);
  else bn_stats_kernel<bf16><<<(D + 31) / 32, 32 * kBnRL, 0, ST(stream)>>>(CBF(x), B, D, out);
  DVGR_CHECK_LAUNCH("bn_stats");
  return 0;
}
extern "C" int DVGR_FN(dvgr_bn_bwd_ex)(const void* dy, const void* x, int x_is_f32, int B, int D, const float* gamma,
                              const float* mean, const float* rstd, int training, void* dx, float* dgamma, float* dbeta,
                              const float* ext_sums, int Btot, int stats_only, void* stream) {
  if (B <= 0 || D <= 0) return 0;
  if (x_is_f32)
    bn_bwd_kernel<float><<<(D + 31) / 32, 32 * kBnRL, 0, ST(stream)>>>(CBF(dy), reinterpret_cast<const float*>(x), B, D, gamma,
                                                                 mean, rstd, training, reinterpret_cast<float*>(dx),
                                                                 dgamma, dbeta, ext_sums, Btot, stats_only);
  else
    bn_bwd_kernel<bf16><<<(D + 31) / 32, 32 * kBnRL, 0, ST(stream)>>>(CBF(dy), CBF(x), B, D, gamma, mean, rstd, training,
                                                                BF(dx), dgamma, dbeta, ext_sums, Btot, stats_only);
  DVGR_CHECK_LAUNCH("bn_bwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_bn_bwd)(const void* dy, const void* x, int x_is_f32, int B, int D, const float* gamma,
                           const float* mean, const float* rstd, int training, void* dx, float* dgamma, float* dbeta,
                           void* stream) {
  return DVGR_FN(dvgr_bn_bwd_ex)(dy, x, x_is_f32, B, D, gamma, mean, rstd, training, dx, dgamma, dbeta, nullptr, B, 0, stream);
}

extern "C" int DVGR_FN(dvgr_cross_entropy_ex)(const float* logits, const long long* answers, int B, int A, float scale,
                                     float* loss_part, void* dlogits, int grad_is_f32, long long ld_d, int* correct,
                                     void* stream) {
  if (B <= 0) return 0;
  if (grad_is_f32)
    ce_kernel<float><<<(B + 7) / 8, 256, 0, ST(stream)>>>(logits, answers, B, A, scale, loss_part,
                                                          reinterpret_cast<float*>(dlogits), ld_d, correct);
  else
    ce_kernel<bf16><<<(B + 7) / 8, 256, 0, ST(stream)>>>(logits, answers, B, A, scale, loss_part, BF(dlogits), ld_d, correct);
  DVGR_CHECK_LAUNCH("cross_entropy");
  return 0;
}
extern "C" int DVGR_FN(dvgr_cross_entropy)(const float* logits, const long long* answers, int B, int A, float scale,
                                  float* loss_part, void* dlogits, long long ld_d, int* correct, void* stream) {
  return DVGR_FN(dvgr_cross_entropy_ex)(logits, answers, B, A, scale, loss_part, dlogits, 0, ld_d, correct, stream);
}

extern "C" int DVGR_FN(dvgr_accuracy_counters)(const float* logits, const long long* answers, int B, int A, const long long* category,
                                      const long long* tokens, long long ld_tok, const int* token_to_cat, int V, int n_cat,
                                      long long* counts, int* preds, void* stream) {
  if (B <= 0) return 0;
  if (!logits || !answers || !counts) return set_error("accuracy_counters: null buffer");
  if (n_cat < 0) return set_error("accuracy_counters: n_cat=%d", n_cat);
  accuracy_counters_kernel<<<(B + 7) / 8, 256, 0, ST(stream)>>>(logits, answers, B, A, category, tokens, ld_tok, token_to_cat,
                                                                V, n_cat, counts, preds);
  DVGR_CHECK_LAUNCH("accuracy_counters");
  return 0;
}

extern "C" int DVGR_FN(dvgr_prep_features_ex)(const void* in, int in_is_bf16, void* out, long long S, int T, int C, int do_tanh,
                                     int time_major, float p, unsigned long long seed, unsigned int drop_stream,
                                     void* stream) {
  if (C % 8 != 0) return set_error("prep_features: C=%d must be a multiple of 8", C);
  const long long n = S * T * (long long)C / 8;
  if (n <= 0) return 0;
  DropoutCfg dc{seed, drop_stream, p, seed_offset_ptr()};
  const GatherCfg g{nullptr, 0, 0, nullptr};
  if (in_is_bf16)
    prep_features_kernel<__nv_bfloat16, false><<<grid_for(n, 256, 148 * 32), 256, 0, ST(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(in), BF(out), S, T, C, do_tanh, time_major, dc, g);
  else
    prep_features_kernel<float, false><<<grid_for(n, 256, 148 * 32), 256, 0, ST(stream)>>>(reinterpret_cast<const float*>(in), BF(out), S, T, C,
                                                                                    do_tanh, time_major, dc, g);
  DVGR_CHECK_LAUNCH("prep_features");
  return 0;
}

extern "C" int DVGR_FN(dvgr_prep_features_gather)(const void* store, int store_is_bf16, long long V, int N, const int* rows,
                                                  int B, void* out, int T, int C, int do_tanh, int time_major, float p,
                                                  unsigned long long seed, unsigned int drop_stream, int* err, void* stream) {
  if (C % 8 != 0) return set_error("prep_features_gather: C=%d must be a multiple of 8", C);
  if (V < 0 || N <= 0 || T <= 0 || B < 0) return set_error("prep_features_gather: V=%lld N=%d T=%d B=%d", V, N, T, B);
  if (!store || !rows || !out || !err) return set_error("prep_features_gather: null buffer");
  const long long slab8 = (long long)N * T * (C / 8);
  if (slab8 > 0x7fffffffLL) return set_error("prep_features_gather: N*T*C/8=%lld exceeds 2^31", slab8);
  const long long S = (long long)B * N;
  const long long n = S * T * (long long)C / 8;
  if (n <= 0) return 0;
  DropoutCfg dc{seed, drop_stream, p, seed_offset_ptr()};
  const GatherCfg g{rows, V, (int)slab8, err};
  if (store_is_bf16)
    prep_features_kernel<__nv_bfloat16, true><<<grid_for(n, 256, 148 * 32), 256, 0, ST(stream)>>>(
        reinterpret_cast<const __nv_bfloat16*>(store), BF(out), S, T, C, do_tanh, time_major, dc, g);
  else
    prep_features_kernel<float, true><<<grid_for(n, 256, 148 * 32), 256, 0, ST(stream)>>>(
        reinterpret_cast<const float*>(store), BF(out), S, T, C, do_tanh, time_major, dc, g);
  DVGR_CHECK_LAUNCH("prep_features_gather");
  return 0;
}

extern "C" int DVGR_FN(dvgr_prep_features)(const float* in, void* out, long long S, int T, int C, int do_tanh, int time_major,
                                  float p, unsigned long long seed, unsigned int drop_stream, void* stream) {
  return DVGR_FN(dvgr_prep_features_ex)(in, 0, out, S, T, C, do_tanh, time_major, p, seed, drop_stream, stream);
}

extern "C" int DVGR_FN(dvgr_cast_rows)(const float* in, long long ld_in, void* out, long long ld_out, int rows, int cols,
                              int out_cols, int lstm_H, void* stream) {
  const long long n = (long long)rows * out_cols;
  if (n <= 0) return 0;
  if (lstm_H > 0 && rows != 4 * lstm_H) return set_error("cast_rows: rows=%d != 4*H=%d", rows, 4 * lstm_H);
  cast_rows_kernel<<<grid_for(n), 256, 0, ST(stream)>>>(in, ld_in, BF(out), ld_out, rows, cols, out_cols, lstm_H);
  DVGR_CHECK_LAUNCH("cast_rows");
  return 0;
}

extern "C" int DVGR_FN(dvgr_split3)(const float* in, long long ld_in, int rows, int cols, void* out, long long ld_out, void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  if (!in || !out) return set_error("split3: null buffer");
  if (ld_out % 8 != 0 || ld_out < cols) return set_error("split3: ld_out=%lld must be a multiple of 8 and >= cols=%d", ld_out, cols);
  const long long n = (long long)rows * (ld_out / 8);
  split3_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, ST(stream)>>>(in, ld_in, rows, cols, BF(out), ld_out, (long long)rows * ld_out);
  DVGR_CHECK_LAUNCH("split3");
  return 0;
}

extern "C" int DVGR_FN(dvgr_dropout)(const void* in, void* out, long long n, float p, unsigned long long seed,
                            unsigned int drop_stream, void* stream) {
  if (n % 8 != 0) return set_error("dropout: n=%lld must be a multiple of 8", n);
  if (n <= 0) return 0;
  DropoutCfg dc{seed, drop_stream, p, seed_offset_ptr()};
  dropout_kernel<<<grid_for(n / 8), 256, 0, ST(stream)>>>(CBF(in), BF(out), n / 8, dc);
  DVGR_CHECK_LAUNCH("dropout");
  return 0;
}


extern "C" int DVGR_FN(dvgr_dropout_multi)(const void* const* in, void* const* out, const unsigned int* drop_streams, int n_copies,
                                  long long n, float p, unsigned long long seed, void* stream) {
  if (n % 8 != 0) return set_error("dropout_multi: n=%lld must be a multiple of 8", n);
  if (n_copies < 1 || n_copies > 4) return set_error("dropout_multi: n_copies=%d out of range [1,4]", n_copies);
  if (n <= 0) return 0;
  DropMulti m;
  memset(&m, 0, sizeof(m));
  for (int i = 0; i < n_copies; ++i) {
    if (!in[i] || !out[i]) return set_error("dropout_multi: null pointer for copy %d", i);
    m.in[i] = CBF(in[i]); m.out[i] = BF(out[i]); m.stream[i] = drop_streams[i];
  }
  DropoutCfg dc{seed, 0u, p, seed_offset_ptr()};
  dropout_multi_kernel<<<dim3(grid_for(n / 8, 256, 148 * 4), n_copies), 256, 0, ST(stream)>>>(m, n / 8, dc);
  DVGR_CHECK_LAUNCH("dropout_multi");
  return 0;
}

extern "C" int DVGR_FN(dvgr_gat_input_bwd)(const void* const* dxt, const unsigned int* drop_streams, int n_streams, int per_stream,
                                  const void* const* base, void* const* out, long long n, float p, unsigned long long seed,
                                  void* stream) {
  if (n % 8 != 0) return set_error("gat_input_bwd: n=%lld must be a multiple of 8", n);
  if (n_streams < 1 || n_streams > 2 || per_stream < 1 || n_streams * per_stream > 4)
    return set_error("gat_input_bwd: %d streams x %d graphs out of range", n_streams, per_stream);
  if (n <= 0) return 0;
  GatInBwd m;
  memset(&m, 0, sizeof(m));
  m.per_stream = per_stream;
  for (int g = 0; g < n_streams * per_stream; ++g) {
    if (!dxt[g]) return set_error("gat_input_bwd: null gradient for graph %d", g);
    m.dxt[g] = CBF(dxt[g]); m.stream[g] = drop_streams[g];
  }
  for (int s_ = 0; s_ < n_streams; ++s_) {
    if (!out[s_]) return set_error("gat_input_bwd: null output for stream %d", s_);
    m.base[s_] = base ? CBF(base[s_]) : nullptr; m.out[s_] = BF(out[s_]);
  }
  DropoutCfg dc{seed, 0u, p, seed_offset_ptr()};
  gat_input_bwd_kernel<<<dim3(grid_for(n / 8, 256, 148 * 8), n_streams), 256, 0, ST(stream)>>>(m, n / 8, dc);
  DVGR_CHECK_LAUNCH("gat_input_bwd");
  return 0;
}

extern "C" int DVGR_FN(dvgr_embed_fwd)(const long long* tokens, const float* table, int B, int L, int W, int Wp, void* words,
                              void* x_tm, float p, unsigned long long seed, unsigned int drop_stream, void* stream) {
  if (B <= 0 || L <= 0) return 0;
  if (Wp % 8 != 0 || Wp < W) return set_error("embed: Wp=%d must be a multiple of 8 and >= W=%d", Wp, W);
  DropoutCfg dc{seed, drop_stream, p, seed_offset_ptr()};
  embed_fwd_kernel<<<grid_for((long long)B * L * (Wp / 8)), 256, 0, ST(stream)>>>(tokens, table, B, L, W, Wp, BF(words),
                                                                                   BF(x_tm), dc);
  DVGR_CHECK_LAUNCH("embed_fwd");
  return 0;
}
extern "C" int DVGR_FN(dvgr_embed_bwd)(const long long* tokens, const void* words, const void* d_words, const void* d_x_tm, int B,
                              int L, int W, int Wp, float* dtable, float p, unsigned long long seed,
                              unsigned int drop_stream, void* stream) {
  if (B <= 0 || L <= 0) return 0;
  if (Wp % 8 != 0 || Wp < W) return set_error("embed: Wp=%d must be a multiple of 8 and >= W=%d", Wp, W);
  DropoutCfg dc{seed, drop_stream, p, seed_offset_ptr()};
  embed_bwd_kernel<<<grid_for((long long)B * L * (Wp / 8)), 256, 0, ST(stream)>>>(tokens, CBF(words), CBF(d_words),
                                                                                   CBF(d_x_tm), B, L, W, Wp, dtable, dc);
  DVGR_CHECK_LAUNCH("embed_bwd");
  return 0;
}

extern "C" int DVGR_FN(dvgr_cast_rows_grouped)(const float* const* in, const long long* ld_in, void* const* out, const int* rows,
                                      const int* cols, int n, long long ld_out, int out_cols, int lstm_H, void* stream) {
  if (n <= 0) return 0;
  if (n > kMaxCast) return set_error("cast_rows_grouped: n=%d > %d", n, kMaxCast);
  CastGroup G;
  memset(&G, 0, sizeof(G));
  long long most = 0;
  for (int i = 0; i < n; ++i) {
    if (!in[i] || !out[i]) return set_error("cast_rows_grouped: null pointer in problem %d", i);
    if (lstm_H > 0 && rows[i] != 4 * lstm_H) return set_error("cast_rows_grouped: rows=%d != 4*H=%d", rows[i], 4 * lstm_H);
    G.in[i] = in[i]; G.out[i] = BF(out[i]); G.ld_in[i] = ld_in[i]; G.rows[i] = rows[i]; G.cols[i] = cols[i];
    most = std::max(most, (long long)rows[i] * out_cols);
  }
  G.ld_out = ld_out; G.out_cols = out_cols; G.lstm_H = lstm_H;
  if (most <= 0) return 0;
  cast_rows_grouped_kernel<<<dim3(grid_for(most / 8 + 1, 256, 148 * 4), n), 256, 0, ST(stream)>>>(G);
  DVGR_CHECK_LAUNCH("cast_rows_grouped");
  return 0;
}

extern "C" int DVGR_FN(dvgr_lstm_pack_bias)(const float* const* b_ih, const float* const* b_hh, int ndir, int H, float* out,
                                   void* stream) {
  if (ndir < 1 || ndir > 4) return set_error("lstm_pack_bias: ndir=%d out of range [1,4]", ndir);
  BiasGroup G;
  memset(&G, 0, sizeof(G));
  for (int d = 0; d < ndir; ++d) {
    if (!b_ih[d] || !b_hh[d]) return set_error("lstm_pack_bias: null bias for direction %d", d);
    G.b_ih[d] = b_ih[d]; G.b_hh[d] = b_hh[d];
  }
  lstm_pack_bias_kernel<<<dim3((4 * H + 255) / 256, ndir), 256, 0, ST(stream)>>>(G, H, out);
  DVGR_CHECK_LAUNCH("lstm_pack_bias");
  return 0;
}

extern "C" int DVGR_FN(dvgr_lstm_pack_dh)(const void* d_seq, long long ld_seq, int nd_seq, const void* d_last, long long ld_last,
                                 int d_last0, int S, int T, int D, int H, void* dh_seq, void* dh_last, void* stream) {
  if (S <= 0 || T <= 0 || D <= 0) return 0;
  if (H % 8 != 0 || ld_seq % 8 != 0 || ld_last % 8 != 0) return set_error("lstm_pack_dh: H and row strides must be multiples of 8");
  const long long n = (long long)T * D * ((S + 31) / 32) * (H / 8) * 32 + (long long)S * D * (H / 8);
  lstm_pack_dh_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, ST(stream)>>>(CBF(d_seq), ld_seq, nd_seq, CBF(d_last), ld_last,
                                                                         d_last0, S, T, D, H, BF(dh_seq), BF(dh_last));
  DVGR_CHECK_LAUNCH("lstm_pack_dh");
  return 0;
}

extern "C" int DVGR_FN(dvgr_act_bwd)(const void* dy, const void* y, void* out, long long n, int act, int accumulate, float p,
                            unsigned long long seed, unsigned int drop_stream, void* stream) {
  if (n % 8 != 0) return set_error("act_bwd: n=%lld must be a multiple of 8", n);
  if (n <= 0) return 0;
  DropoutCfg dc{seed, drop_stream, p, seed_offset_ptr()};
  act_bwd_kernel<<<grid_for(n / 8), 256, 0, ST(stream)>>>(CBF(dy), CBF(y), BF(out), n / 8, act, accumulate, dc);
  DVGR_CHECK_LAUNCH("act_bwd");
  return 0;
}

// Grouped column sums: out_i[C_i] += sum over rows of in_i[R_i][C_i] for up to kMaxColsum problems in ONE launch (the bias
// gradients of the nn.Linear layers: like their weight gradients nothing reads them before the optimizer, so the autograd
// layer queues them and the engine flushes the queue once per step). One block = (problem, 256-column block, row chunk);
// partial sums are added with fp32 atomics (the order of the chunk contributions is not fixed, as for the split-K wgrads).
namespace {
constexpr int kMaxColsum = 48;
struct ColsumGroup {
  const void* in[kMaxColsum];
  float* out[kMaxColsum];
  long long ld[kMaxColsum];
  int R[kMaxColsum], C[kMaxColsum], is_f32[kMaxColsum], vec_ok[kMaxColsum];
  int block_start[kMaxColsum + 1];      // prefix sums of col_blocks * chunks
  int chunks[kMaxColsum], rows_per_chunk[kMaxColsum];
  int perm_H[kMaxColsum];               // > 0: input column 4*j + g lands at output index g*H + j (LSTM gate de-interleave)
  float* out2[kMaxColsum];              // optional second accumulation target (b_ih and b_hh share one gradient)
  int n;
};

template <typename T>
__device__ __forceinline__ void colsum_group_block(const T* __restrict__ in, long long ld, long long r0, long long r1, int C,
                                                   int cblk, int vec_ok, float* __restrict__ out, int perm_H,
                                                   float* __restrict__ out2) {
  __shared__ float red[8][32][9];
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c0 = (cblk * 32 + cg) * 8;
  float acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.f;
  if (c0 < C) {
    if (vec_ok && c0 + 8 <= C) {
      long long r = r0 + rl;
      for (; r + 24 < r1; r += 32) {
        float f0[8], f1[8], f2[8], f3[8];
        load8g(in + r * ld + c0, f0);
        load8g(in + (r + 8) * ld + c0, f1);
        load8g(in + (r + 16) * ld + c0, f2);
        load8g(in + (r + 24) * ld + c0, f3);
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] += (f0[q] + f1[q]) + (f2[q] + f3[q]);
      }
      for (; r < r1; r += 8) {
        float f0[8];
        load8g(in + r * ld + c0, f0);
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] += f0[q];
      }
    } else {
      for (long long r = r0 + rl; r < r1; r += 8)
        for (int q = 0; q < 8; ++q)
          if (c0 + q < C) acc[q] += ldf<T>(in + r * ld + c0 + q);
    }
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) red[rl][cg][q] = acc[q];
  __syncthreads();
  if (rl == 0 && c0 < C) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float s_ = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s_ += red[k][cg][q];
      if (c0 + q < C) {
        const int c = c0 + q;
        const int o = perm_H > 0 ? (c & 3) * perm_H + (c >> 2) : c;
        atomicAdd(out + o, s_);
        if (out2 != nullptr) atomicAdd(out2 + o, s_);
      }
    }
  }
}

__global__ void __launch_bounds__(256) colsum_grouped_kernel(const __grid_constant__ ColsumGroup G) {
  pdl_trigger();
  int pi = 0;
  while (pi + 1 < G.n && (int)blockIdx.x >= G.block_start[pi + 1]) ++pi;
  const int t = blockIdx.x - G.block_start[pi];
  const int chunk = t % G.chunks[pi], cblk = t / G.chunks[pi];
  const long long r0 = (long long)chunk * G.rows_per_chunk[pi];
  const long long r1 = min((long long)G.R[pi], r0 + G.rows_per_chunk[pi]);
  if (G.is_f32[pi])
    colsum_group_block<float>(reinterpret_cast<const float*>(G.in[pi]), G.ld[pi], r0, r1, G.C[pi], cblk, G.vec_ok[pi], G.out[pi],
                              G.perm_H[pi], G.out2[pi]);
  else
    colsum_group_block<bf16>(reinterpret_cast<const bf16*>(G.in[pi]), G.ld[pi], r0, r1, G.C[pi], cblk, G.vec_ok[pi], G.out[pi],
                             G.perm_H[pi], G.out2[pi]);
}
}  // namespace

extern "C" int DVGR_FN(dvgr_colsum_grouped)(const dvgr_colsum_problem* probs, int n, void* stream) {
  if (n <= 0) return 0;
  if (!probs) return set_error("colsum_grouped: null problem list");
  for (int base = 0; base < n; base += kMaxColsum) {
    const int cnt = n - base < kMaxColsum ? n - base : kMaxColsum;
    ColsumGroup G;
    memset(&G, 0, sizeof(G));
    G.n = cnt;
    int blocks = 0;
    for (int i = 0; i < cnt; ++i) {
      const dvgr_colsum_problem& q = probs[base + i];
      if (!q.in || !q.out || q.R <= 0 || q.C <= 0) return set_error("colsum_grouped: problem %d is empty or null", base + i);
      const int esz = q.in_is_f32 ? 4 : 2;
      G.in[i] = q.in; G.out[i] = q.out; G.ld[i] = q.ld; G.R[i] = (int)q.R; G.C[i] = q.C; G.is_f32[i] = q.in_is_f32;
      G.vec_ok[i] = ((reinterpret_cast<uintptr_t>(q.in) & 15) == 0) && ((q.ld * esz) % 16 == 0);
      G.perm_H[i] = q.perm_H; G.out2[i] = q.out2;
      if (q.perm_H > 0 && q.C != 4 * q.perm_H) return set_error("colsum_grouped: problem %d: C=%d != 4*perm_H", base + i, q.C);
      long long chunks = (q.R + 255) / 256;          // >= 256 rows per chunk: few atomics per output element
      if (chunks > 64) chunks = 64;
      G.chunks[i] = (int)chunks;
      G.rows_per_chunk[i] = (int)((q.R + chunks - 1) / chunks);
      G.block_start[i] = blocks;
      blocks += ((q.C + 255) / 256) * (int)chunks;
    }
    G.block_start[cnt] = blocks;
    colsum_grouped_kernel<<<blocks, 256, 0, ST(stream)>>>(G);
    DVGR_CHECK_LAUNCH("colsum_grouped");
  }
  return 0;
}

// dst[i] (+)= src[i] for up to kMaxSegs small fp32 segments in ONE launch (one block per segment). accumulate: the gradient
// accumulation of the many tiny parameters of a DualVGR unit (per-head attention vectors and biases), which autograd would
// otherwise perform with one elementwise launch per parameter (~170 launches of ~2 us per train step); copy: gathering those
// parameters into the packed per-graph operands of the GAT kernels (instead of ~25 torch.cat launches per layer).
namespace {
constexpr int kMaxSegs = 128;
struct SegList {
  float* dst[kMaxSegs];
  const float* src[kMaxSegs];
  int n[kMaxSegs];
};
__global__ void scatter_kernel(const SegList L, int accumulate) {
  pdl_trigger();
  float* d = L.dst[blockIdx.x];
  const float* s = L.src[blockIdx.x];
  for (int i = threadIdx.x; i < L.n[blockIdx.x]; i += blockDim.x) d[i] = accumulate ? d[i] + s[i] : s[i];
}
}  // namespace

extern "C" int DVGR_FN(dvgr_scatter)(const dvgr_seg* segs, int n_segs, int accumulate, void* stream) {
  if (n_segs <= 0) return 0;
  if (!segs) return set_error("scatter: null segment list");
  for (int base = 0; base < n_segs; base += kMaxSegs) {
    SegList L;
    const int cnt = n_segs - base < kMaxSegs ? n_segs - base : kMaxSegs;
    for (int i = 0; i < cnt; ++i) {
      if (!segs[base + i].dst || !segs[base + i].src) return set_error("scatter: segment %d has a null pointer", base + i);
      L.dst[i] = segs[base + i].dst; L.src[i] = segs[base + i].src; L.n[i] = segs[base + i].n;
    }
    scatter_kernel<<<cnt, 128, 0, ST(stream)>>>(L, accumulate);
    DVGR_CHECK_LAUNCH("scatter");
  }
  return 0;
}

extern "C" int DVGR_FN(dvgr_add)(void* a, const void* b, long long n, void* stream) {
  if (n % 8 != 0) return set_error("add: n=%lld must be a multiple of 8", n);
  if (n <= 0) return 0;
  add_kernel<<<grid_for(n / 8), 256, 0, ST(stream)>>>(BF(a), CBF(b), n / 8);
  DVGR_CHECK_LAUNCH("add");
  return 0;
}

static inline long long colsum_chunks(long long R) {
  long long chunks = (R + 63) / 64;          // >= 64 rows (8 per row lane) per chunk
  if (chunks > 256) chunks = 256;
  if (chunks < 1) chunks = 1;
  return chunks;
}

extern "C" long long DVGR_FN(dvgr_colsum_workspace)(long long R, int C) { return colsum_chunks(R) * C; }

extern "C" int DVGR_FN(dvgr_colsum_batched)(const void* in, int in_is_f32, long long ld, long long in_batch, long long R, int C,
                                   int batch, float* workspace, float* out, long long out_batch, int accumulate,
                                   float scale, void* stream) {
  if (C <= 0 || batch <= 0) return 0;
  const long long chunks = colsum_chunks(R);
  const int rpc = (int)((R + chunks - 1) / chunks);
  dim3 grid((C + 255) / 256, (unsigned)chunks, (unsigned)batch);
  const int esz = in_is_f32 ? 4 : 2;
  const int vec_ok = ((reinterpret_cast<uintptr_t>(in) & 15) == 0) && ((ld * esz) % 16 == 0) && ((in_batch * esz) % 16 == 0);
  if (in_is_f32)
    colsum_partial_kernel<float><<<grid, 256, 0, ST(stream)>>>(reinterpret_cast<const float*>(in), ld, R, C, rpc, workspace, vec_ok, in_batch);
  else
    colsum_partial_kernel<bf16><<<grid, 256, 0, ST(stream)>>>(CBF(in), ld, R, C, rpc, workspace, vec_ok, in_batch);
  DVGR_CHECK_LAUNCH("colsum_partial");
  colsum_final_kernel<<<dim3((C + 31) / 32, 1, batch), 256, 0, ST(stream)>>>(workspace, (int)chunks, C, out, accumulate, scale, out_batch);
  DVGR_CHECK_LAUNCH("colsum_final");
  return 0;
}

extern "C" int DVGR_FN(dvgr_colsum)(const void* in, int in_is_f32, long long ld, long long R, int C, float* workspace, float* out,
                           int accumulate, float scale, void* stream) {
  return DVGR_FN(dvgr_colsum_batched)(in, in_is_f32, ld, 0, R, C, 1, workspace, out, 0, accumulate, scale, stream);
}
