// Kernels of SASRecModel (models/sequential/sasrec.py; SURVEY.md section 8(f) row N3): the satisfied-only history (item | category,
// S = 20 or 40 wide) plus a learned position table goes through two pre-LN self-attention blocks with DENSE biased Q / K / V projections
// (tf.layers.dense, sasrec.py:268-270 - PAMRec's time-aware tables replace exactly these), one head, key mask = satisfied_mask, no
// query mask, no causality (sasrec.py:89); the state at the last satisfied position joins the target in front of one tower.
//
// One thread per token holds a token's S-vectors in registers: every token-local step runs with the S x S matrices in shared memory
// (all lanes read the same weight: broadcast), attention is one thread per query row (forward, dQ) or per key row (dK, dV) over the
// sample's rows in shared memory.  Weight gradients are reductions over tokens and run on the grouped dW kernel of kernels_head.cu;
// this file stores the operands those GEMMs need.
#include "head_tiles.cuh"

namespace pamrec {

// The model width S = item + cate embedding width: 20 (config/sasrec.yaml as shipped) or 40 (the reference's 32 / 8).  Every kernel
// is a template on S; the launchers pick the instantiation once per launch.
template <int S> struct SasW { static constexpr int value = S; };
template <typename F> static void sas_widths(int S, F f) {
  if (S == 40) f(SasW<40>{});
  else f(SasW<20>{});
}
// 1 / sqrt(S)   (sasrec.py:284)
template <int S> __device__ __forceinline__ float sas_scale() { return S == 40 ? 0.15811388300841897f : 0.22360679774997896f; }

template <int S>
__device__ __forceinline__ void sas_load(const float* __restrict__ p, float (&x)[S]) {
#pragma unroll
  for (int c = 0; c < S / 4; ++c) {
    const float4 v = ld4(p + 4 * c);
    x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
  }
}
template <int S>
__device__ __forceinline__ void sas_store(float* __restrict__ p, const float (&x)[S]) {
#pragma unroll
  for (int c = 0; c < S / 4; ++c) st4(p + 4 * c, make_float4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]));
}
// sasrec.py:144-170 (normalize): population variance, eps 1e-8 inside the square root
template <int S>
__device__ __forceinline__ void sas_ln(const float (&x)[S], const float* __restrict__ beta, const float* __restrict__ gamma, float (&xh)[S],
                                       float (&y)[S], float& rstd) {
  float mean = 0.f;
#pragma unroll
  for (int i = 0; i < S; ++i) mean += x[i];
  mean *= (1.0f / S);
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < S; ++i) { const float d = x[i] - mean; var = fmaf(d, d, var); }
  var *= (1.0f / S);
  rstd = 1.0f / sqrtf(var + kLnEps);
#pragma unroll
  for (int i = 0; i < S; ++i) { xh[i] = (x[i] - mean) * rstd; y[i] = fmaf(gamma[i], xh[i], beta[i]); }
}
// gradient of LN: dx = rstd * (g - mean(g) - xh * mean(g * xh)),  g = dy * gamma
template <int S>
__device__ __forceinline__ void sas_ln_bwd(const float (&dy)[S], const float (&xh)[S], const float* __restrict__ gamma, float rstd, float (&dx)[S]) {
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < S; ++i) { const float g = dy[i] * gamma[i]; s1 += g; s2 = fmaf(g, xh[i], s2); }
  s1 *= (1.0f / S); s2 *= (1.0f / S);
#pragma unroll
  for (int i = 0; i < S; ++i) dx[i] = rstd * (dy[i] * gamma[i] - s1 - xh[i] * s2);
}
// out[j] = sum_i a[i] W[i][j]   (W row-major [S][S] in shared memory; every lane reads the same address)
template <int S>
__device__ __forceinline__ void sas_matvec(const float (&a)[S], const float* __restrict__ W, float (&out)[S]) {
#pragma unroll
  for (int j = 0; j < S; ++j) out[j] = 0.f;
#pragma unroll
  for (int i = 0; i < S; ++i) {
    const float ai = a[i];
#pragma unroll
    for (int c = 0; c < S / 4; ++c) {
      const float4 w = ld4(W + i * S + 4 * c);
      out[4 * c] = fmaf(ai, w.x, out[4 * c]); out[4 * c + 1] = fmaf(ai, w.y, out[4 * c + 1]);
      out[4 * c + 2] = fmaf(ai, w.z, out[4 * c + 2]); out[4 * c + 3] = fmaf(ai, w.w, out[4 * c + 3]);
    }
  }
}
// out[i] = sum_j a[j] W[i][j]   (the transposed product of the backward pass)
template <int S>
__device__ __forceinline__ void sas_matvec_t(const float (&a)[S], const float* __restrict__ W, float (&out)[S]) {
#pragma unroll
  for (int i = 0; i < S; ++i) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < S / 4; ++c) {
      const float4 w = ld4(W + i * S + 4 * c);
      s = fmaf(a[4 * c], w.x, s); s = fmaf(a[4 * c + 1], w.y, s); s = fmaf(a[4 * c + 2], w.z, s); s = fmaf(a[4 * c + 3], w.w, s);
    }
    out[i] = s;
  }
}
// CTA-wide sums of two per-thread vectors of S (LN parameter gradients), added to global memory by 2 S threads
template <int S>
__device__ __forceinline__ void sas_reduce_ln_grads(float (&dg)[S], float (&db)[S], float* __restrict__ g_gamma, float* __restrict__ g_beta,
                                                    float* red /* [warps][2 S] */) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int i = 0; i < S; ++i) { dg[i] = warp_sum(dg[i]); db[i] = warp_sum(db[i]); }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < S; ++i) { red[w * 2 * S + i] = dg[i]; red[w * 2 * S + S + i] = db[i]; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * S) {
    float s = 0.f;
    for (int k = 0; k < nw; ++k) s += red[k * 2 * S + threadIdx.x];
    if (s != 0.f) atomicAdd(threadIdx.x < S ? g_gamma + threadIdx.x : g_beta + (threadIdx.x - S), s);
  }
}

// ------------------------------------------------------------------------------------------ embedding
// seq0[n] = history token + position row (sasrec.py:61-64)
template <int S>
__global__ void __launch_bounds__(256) k_sas_embed(const float* __restrict__ h, const float* __restrict__ pos, float* __restrict__ x0,
                                                   int64_t N, int T) {
  constexpr int CH = S / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * CH) return;
  const int64_t n = i / CH;
  const int c = (int)(i % CH), t = (int)(n % T);
  const float4 a = ld4(h + n * S + 4 * c), p = ld4(pos + t * S + 4 * c);
  st4(x0 + n * S + 4 * c, make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w));
}
void launch_sas_embed(const float* h, const float* pos, float* x0, int B, int T, int S, cudaStream_t st) { PAMREC_PROF("sas_embed", 1, st);
  if (B == 0) return;
  const int64_t N = (int64_t)B * T;
  sas_widths(S, [&](auto w) {
    constexpr int S_ = decltype(w)::value;
    k_sas_embed<S_><<<(unsigned)((N * (S_ / 4) + 255) / 256), 256, 0, st>>>(h, pos, x0, N, T);
  });
}

// ------------------------------------------------------------------------------------------ projections
// q_in = LN(x);  Q = q_in Wq + bq,  K = x Wk + bk,  V = x Wv + bv   (sasrec.py:89-90, 268-270).  xq = q_in | x is kept: it is the
// left operand of the three weight-gradient GEMMs.  W = [Wq | Wk | Wv] (3 x S^2), bias = [bq | bk | bv].
template <int S>
__global__ void __launch_bounds__(128)
k_sas_proj_fwd(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ bias, const float* __restrict__ ln_beta,
               const float* __restrict__ ln_gamma, float* __restrict__ XQ, float* __restrict__ QKV, int64_t N) {
  constexpr int SS = S * S;
  __shared__ __align__(16) float sw[3 * SS + 3 * S + 2 * S];
  for (int i = threadIdx.x; i < 3 * SS; i += blockDim.x) sw[i] = W[i];
  for (int i = threadIdx.x; i < 3 * S; i += blockDim.x) sw[3 * SS + i] = bias[i];
  if (threadIdx.x < S) { sw[3 * SS + 3 * S + threadIdx.x] = ln_beta[threadIdx.x]; sw[3 * SS + 4 * S + threadIdx.x] = ln_gamma[threadIdx.x]; }
  __syncthreads();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float x[S], xh[S], q[S], o[S], rstd;
  sas_load(X + n * S, x);
  sas_ln(x, sw + 3 * SS + 3 * S, sw + 3 * SS + 4 * S, xh, q, rstd);
  sas_store(XQ + n * 2 * S, q);
  sas_store(XQ + n * 2 * S + S, x);
  sas_matvec(q, sw, o);
#pragma unroll
  for (int j = 0; j < S; ++j) o[j] += sw[3 * SS + j];
  sas_store(QKV + n * 3 * S, o);
  sas_matvec(x, sw + SS, o);
#pragma unroll
  for (int j = 0; j < S; ++j) o[j] += sw[3 * SS + S + j];
  sas_store(QKV + n * 3 * S + S, o);
  sas_matvec(x, sw + 2 * SS, o);
#pragma unroll
  for (int j = 0; j < S; ++j) o[j] += sw[3 * SS + 2 * S + j];
  sas_store(QKV + n * 3 * S + 2 * S, o);
}
void launch_sas_proj_fwd(const float* X, const float* W, const float* bias, const float* ln_beta, const float* ln_gamma, float* XQ,
                         float* QKV, int64_t N, int S, cudaStream_t st) { PAMREC_PROF("sas_proj_fwd", 1, st);
  if (N == 0) return;
  sas_widths(S, [&](auto w) {
    k_sas_proj_fwd<decltype(w)::value><<<(unsigned)((N + 127) / 128), 128, 0, st>>>(X, W, bias, ln_beta, ln_gamma, XQ, QKV, N);
  });
}

// d q_in = dQ Wq^T + dY (the residual on the queries);  dX = dK Wk^T + dV Wv^T + LN'(d q_in);  LN parameter gradients
template <int S>
__global__ void __launch_bounds__(128)
k_sas_proj_bwd(const float* __restrict__ XQ, const float* __restrict__ dQKV, const float* __restrict__ dY, const float* __restrict__ W,
               const float* __restrict__ ln_gamma, float* __restrict__ dX, float* __restrict__ g_gamma, float* __restrict__ g_beta, int64_t N) {
  constexpr int SS = S * S;
  __shared__ __align__(16) float sw[3 * SS + S];
  __shared__ float red[4 * 2 * S];
  for (int i = threadIdx.x; i < 3 * SS; i += blockDim.x) sw[i] = W[i];
  if (threadIdx.x < S) sw[3 * SS + threadIdx.x] = ln_gamma[threadIdx.x];
  __syncthreads();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float dg[S], db[S];
#pragma unroll
  for (int i = 0; i < S; ++i) { dg[i] = 0.f; db[i] = 0.f; }
  if (n < N) {
    float x[S], g[S], acc[S], dqin[S], dx[S];
    sas_load(dQKV + n * 3 * S, g);
    sas_matvec_t(g, sw, dqin);
    sas_load(dY + n * S, g);
#pragma unroll
    for (int i = 0; i < S; ++i) dqin[i] += g[i];
    sas_load(dQKV + n * 3 * S + S, g);
    sas_matvec_t(g, sw + SS, acc);
    sas_load(dQKV + n * 3 * S + 2 * S, g);
    sas_matvec_t(g, sw + 2 * SS, dx);
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] += dx[i];
    // LN statistics of x again (xq holds q_in = gamma * xhat + beta; x itself is the second half)
    sas_load(XQ + n * 2 * S + S, x);
    float mean = 0.f;
#pragma unroll
    for (int i = 0; i < S; ++i) mean += x[i];
    mean *= (1.0f / S);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < S; ++i) { const float d = x[i] - mean; var = fmaf(d, d, var); }
    var *= (1.0f / S);
    const float rstd = 1.0f / sqrtf(var + kLnEps);
    float xh[S];
#pragma unroll
    for (int i = 0; i < S; ++i) { xh[i] = (x[i] - mean) * rstd; dg[i] = dqin[i] * xh[i]; db[i] = dqin[i]; }
    sas_ln_bwd(dqin, xh, sw + 3 * SS, rstd, dx);
#pragma unroll
    for (int i = 0; i < S; ++i) dx[i] += acc[i];
    sas_store(dX + n * S, dx);
  }
  sas_reduce_ln_grads(dg, db, g_gamma, g_beta, red);
}
void launch_sas_proj_bwd(const float* XQ, const float* dQKV, const float* dY, const float* W, const float* ln_gamma, float* dX,
                         float* g_gamma, float* g_beta, int64_t N, int S, cudaStream_t st) { PAMREC_PROF("sas_proj_bwd", 1, st);
  if (N == 0) return;
  sas_widths(S, [&](auto w) {
    k_sas_proj_bwd<decltype(w)::value><<<(unsigned)((N + 127) / 128), 128, 0, st>>>(XQ, dQKV, dY, W, ln_gamma, dX, g_gamma, g_beta, N);
  });
}

// ------------------------------------------------------------------------------------------ attention
// y = softmax_t(mask_t ? q . k_t / sqrt(S) : -(2^32)+1) V + q_in   (sasrec.py:281-324); ML = (row maximum, row sum)
template <int S>
__global__ void __launch_bounds__(128)
k_sas_attn_fwd(const float* __restrict__ QKV, const float* __restrict__ XQ, const int* __restrict__ mask, float* __restrict__ Y,
               float* __restrict__ ML, int T) {
  constexpr int CH = S / 4;
  const float scale = sas_scale<S>();
  extern __shared__ __align__(16) float sm[];
  float* Ks = sm;                       // [T][S]
  float* Vs = Ks + T * S;               // [T][S]
  int* Ms = reinterpret_cast<int*>(Vs + T * S);
  const int b = blockIdx.x;
  const int64_t base = (int64_t)b * T;
  for (int i = threadIdx.x; i < T * CH; i += blockDim.x) {
    const int t = i / CH, c = i % CH;
    st4(Ks + t * S + 4 * c, ld4(QKV + (base + t) * 3 * S + S + 4 * c));
    st4(Vs + t * S + 4 * c, ld4(QKV + (base + t) * 3 * S + 2 * S + 4 * c));
  }
  for (int t = threadIdx.x; t < T; t += blockDim.x) Ms[t] = mask[base + t];
  __syncthreads();
  for (int tq = threadIdx.x; tq < T; tq += blockDim.x) {
    float q[S], acc[S];
    sas_load(QKV + (base + tq) * 3 * S, q);
    float m = -INFINITY;
    for (int t = 0; t < T; ++t) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < S; ++i) s = fmaf(q[i], Ks[t * S + i], s);
      s = Ms[t] == 1 ? s * scale : kMaskNeg;
      m = fmaxf(m, s);
    }
    float l = 0.f;
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] = 0.f;
    for (int t = 0; t < T; ++t) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < S; ++i) s = fmaf(q[i], Ks[t * S + i], s);
      s = Ms[t] == 1 ? s * scale : kMaskNeg;
      const float e = expf(s - m);
      l += e;
#pragma unroll
      for (int i = 0; i < S; ++i) acc[i] = fmaf(e, Vs[t * S + i], acc[i]);
    }
    float qin[S];
    sas_load(XQ + (base + tq) * 2 * S, qin);
    const float inv = 1.0f / l;
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] = fmaf(acc[i], inv, qin[i]);
    sas_store(Y + (base + tq) * S, acc);
    ML[(base + tq) * 2] = m;
    ML[(base + tq) * 2 + 1] = l;
  }
}

// dQ per query row; also Dq = dY . (Y - q_in) = sum_t p_t dP_t, which the key pass needs
template <int S>
__global__ void __launch_bounds__(128)
k_sas_attn_bwd_q(const float* __restrict__ QKV, const float* __restrict__ XQ, const float* __restrict__ Y, const float* __restrict__ dY,
                 const float* __restrict__ ML, const int* __restrict__ mask, float* __restrict__ dQKV, float* __restrict__ Dq, int T) {
  constexpr int CH = S / 4;
  const float scale = sas_scale<S>();
  extern __shared__ __align__(16) float sm[];
  float* Ks = sm;
  float* Vs = Ks + T * S;
  int* Ms = reinterpret_cast<int*>(Vs + T * S);
  const int b = blockIdx.x;
  const int64_t base = (int64_t)b * T;
  for (int i = threadIdx.x; i < T * CH; i += blockDim.x) {
    const int t = i / CH, c = i % CH;
    st4(Ks + t * S + 4 * c, ld4(QKV + (base + t) * 3 * S + S + 4 * c));
    st4(Vs + t * S + 4 * c, ld4(QKV + (base + t) * 3 * S + 2 * S + 4 * c));
  }
  for (int t = threadIdx.x; t < T; t += blockDim.x) Ms[t] = mask[base + t];
  __syncthreads();
  for (int tq = threadIdx.x; tq < T; tq += blockDim.x) {
    float q[S], dy[S], tmp[S], dq[S];
    sas_load(QKV + (base + tq) * 3 * S, q);
    sas_load(dY + (base + tq) * S, dy);
    sas_load(Y + (base + tq) * S, tmp);
    float qin[S];
    sas_load(XQ + (base + tq) * 2 * S, qin);
    float D = 0.f;
#pragma unroll
    for (int i = 0; i < S; ++i) D = fmaf(dy[i], tmp[i] - qin[i], D);
    const float m = ML[(base + tq) * 2], inv = 1.0f / ML[(base + tq) * 2 + 1];
#pragma unroll
    for (int i = 0; i < S; ++i) dq[i] = 0.f;
    for (int t = 0; t < T; ++t) {
      if (Ms[t] != 1) continue;                    // tf.where: no gradient reaches the score of a masked key
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int i = 0; i < S; ++i) { s = fmaf(q[i], Ks[t * S + i], s); dp = fmaf(dy[i], Vs[t * S + i], dp); }
      const float p = expf(s * scale - m) * inv;
      const float ds = p * (dp - D) * scale;
#pragma unroll
      for (int i = 0; i < S; ++i) dq[i] = fmaf(ds, Ks[t * S + i], dq[i]);
    }
    sas_store(dQKV + (base + tq) * 3 * S, dq);
    Dq[base + tq] = D;
  }
}
// dK, dV per key row (sum over the queries of the sample)
template <int S>
__global__ void __launch_bounds__(128)
k_sas_attn_bwd_kv(const float* __restrict__ QKV, const float* __restrict__ dY, const float* __restrict__ ML, const float* __restrict__ Dq,
                  const int* __restrict__ mask, float* __restrict__ dQKV, int T) {
  constexpr int CH = S / 4;
  const float scale = sas_scale<S>();
  extern __shared__ __align__(16) float sm[];
  float* Qs = sm;                       // [T][S]
  float* Gs = Qs + T * S;               // dY [T][S]
  float* Ss = Gs + T * S;               // [T][3]  m, 1 / l, D
  const int b = blockIdx.x;
  const int64_t base = (int64_t)b * T;
  for (int i = threadIdx.x; i < T * CH; i += blockDim.x) {
    const int t = i / CH, c = i % CH;
    st4(Qs + t * S + 4 * c, ld4(QKV + (base + t) * 3 * S + 4 * c));
    st4(Gs + t * S + 4 * c, ld4(dY + (base + t) * S + 4 * c));
  }
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    Ss[t * 3] = ML[(base + t) * 2]; Ss[t * 3 + 1] = 1.0f / ML[(base + t) * 2 + 1]; Ss[t * 3 + 2] = Dq[base + t];
  }
  __syncthreads();
  for (int tk = threadIdx.x; tk < T; tk += blockDim.x) {
    float k[S], v[S], dk[S], dv[S];
    sas_load(QKV + (base + tk) * 3 * S + S, k);
    sas_load(QKV + (base + tk) * 3 * S + 2 * S, v);
    const bool live = mask[base + tk] == 1;
#pragma unroll
    for (int i = 0; i < S; ++i) { dk[i] = 0.f; dv[i] = 0.f; }
    for (int tq = 0; tq < T; ++tq) {
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int i = 0; i < S; ++i) { s = fmaf(Qs[tq * S + i], k[i], s); dp = fmaf(Gs[tq * S + i], v[i], dp); }
      s = live ? s * scale : kMaskNeg;
      const float p = expf(s - Ss[tq * 3]) * Ss[tq * 3 + 1];       // a masked key still has weight 1 / T in a row without any live key
#pragma unroll
      for (int i = 0; i < S; ++i) dv[i] = fmaf(p, Gs[tq * S + i], dv[i]);
      if (live) {
        const float ds = p * (dp - Ss[tq * 3 + 2]) * scale;
#pragma unroll
        for (int i = 0; i < S; ++i) dk[i] = fmaf(ds, Qs[tq * S + i], dk[i]);
      }
    }
    sas_store(dQKV + (base + tk) * 3 * S + S, dk);
    sas_store(dQKV + (base + tk) * 3 * S + 2 * S, dv);
  }
}
// dynamic shared memory of the three attention kernels: K | V | mask (forward, dQ) or Q | dY | (m, 1 / l, D) (dK, dV)
static size_t sas_attn_smem(int T, int S, bool kv) { return (size_t)T * (2 * S + (kv ? 3 : 1)) * sizeof(float); }
// At S = 40 and T = 256 the tiles need 81 / 83 KB: opt in to more than 48 KB of dynamic shared memory (called by pamrec_bind)
int init_sas_kernels(int max_T) {
  int rc = 0;
  sas_widths(40, [&](auto w) {
    constexpr int S = decltype(w)::value;
    const void* fns[3] = {(const void*)k_sas_attn_fwd<S>, (const void*)k_sas_attn_bwd_q<S>, (const void*)k_sas_attn_bwd_kv<S>};
    for (int i = 0; i < 3; ++i) {
      const size_t bytes = sas_attn_smem(max_T, S, i == 2);
      if (bytes > 48 * 1024 && cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) rc = -1;
    }
  });
  return rc;
}
void launch_sas_attn_fwd(const float* QKV, const float* XQ, const int* mask, float* Y, float* ML, int B, int T, int S, cudaStream_t st) {
  PAMREC_PROF("sas_attn_fwd", 1, st);
  if (B == 0) return;
  sas_widths(S, [&](auto w) {
    constexpr int S_ = decltype(w)::value;
    k_sas_attn_fwd<S_><<<B, 128, sas_attn_smem(T, S_, false), st>>>(QKV, XQ, mask, Y, ML, T);
  });
}
void launch_sas_attn_bwd(const float* QKV, const float* XQ, const float* Y, const float* dY, const float* ML, const int* mask, float* dQKV,
                         float* Dq, int B, int T, int S, cudaStream_t st) { PAMREC_PROF("sas_attn_bwd", 2, st);
  if (B == 0) return;
  sas_widths(S, [&](auto w) {
    constexpr int S_ = decltype(w)::value;
    k_sas_attn_bwd_q<S_><<<B, 128, sas_attn_smem(T, S_, false), st>>>(QKV, XQ, Y, dY, ML, mask, dQKV, Dq, T);
    k_sas_attn_bwd_kv<S_><<<B, 128, sas_attn_smem(T, S_, true), st>>>(QKV, dY, ML, Dq, mask, dQKV, T);
  });
}

// ------------------------------------------------------------------------------------------ point-wise feed forward
// f = LN_1(y);  hpre = f W1 + b1;  out = relu(hpre) W2 + b2 + f   (sasrec.py:127-141; the residual is on the normalised input)
template <int S>
__global__ void __launch_bounds__(128)
k_sas_ffn_fwd(const float* __restrict__ Y, const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
              const float* __restrict__ b2, const float* __restrict__ ln_beta, const float* __restrict__ ln_gamma, float* __restrict__ F,
              float* __restrict__ HPRE, float* __restrict__ OUT, int64_t N) {
  constexpr int SS = S * S;
  __shared__ __align__(16) float sw[2 * SS + 4 * S];
  for (int i = threadIdx.x; i < SS; i += blockDim.x) { sw[i] = W1[i]; sw[SS + i] = W2[i]; }
  if (threadIdx.x < S) {
    sw[2 * SS + threadIdx.x] = b1[threadIdx.x]; sw[2 * SS + S + threadIdx.x] = b2[threadIdx.x];
    sw[2 * SS + 2 * S + threadIdx.x] = ln_beta[threadIdx.x]; sw[2 * SS + 3 * S + threadIdx.x] = ln_gamma[threadIdx.x];
  }
  __syncthreads();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float y[S], xh[S], f[S], h[S], o[S], rstd;
  sas_load(Y + n * S, y);
  sas_ln(y, sw + 2 * SS + 2 * S, sw + 2 * SS + 3 * S, xh, f, rstd);
  sas_store(F + n * S, f);
  sas_matvec(f, sw, h);
#pragma unroll
  for (int j = 0; j < S; ++j) h[j] += sw[2 * SS + j];
  sas_store(HPRE + n * S, h);
#pragma unroll
  for (int j = 0; j < S; ++j) h[j] = fmaxf(h[j], 0.f);
  sas_matvec(h, sw + SS, o);
#pragma unroll
  for (int j = 0; j < S; ++j) o[j] += sw[2 * SS + S + j] + f[j];
  sas_store(OUT + n * S, o);
}
void launch_sas_ffn_fwd(const float* Y, const float* W1, const float* b1, const float* W2, const float* b2, const float* ln_beta,
                        const float* ln_gamma, float* F, float* HPRE, float* OUT, int64_t N, int S, cudaStream_t st) {
  PAMREC_PROF("sas_ffn_fwd", 1, st);
  if (N == 0) return;
  sas_widths(S, [&](auto w) {
    k_sas_ffn_fwd<decltype(w)::value><<<(unsigned)((N + 127) / 128), 128, 0, st>>>(Y, W1, b1, W2, b2, ln_beta, ln_gamma, F, HPRE, OUT, N);
  });
}

// d hid = dOut W2^T;  d hpre = [hpre > 0] d hid;  d f = dOut + d hpre W1^T;  dY = LN_1'(d f);  HID = relu(hpre) and DHPRE are kept for
// the weight-gradient GEMMs (dW2 = HID^T dOut, dW1 = F^T DHPRE)
template <int S>
__global__ void __launch_bounds__(128)
k_sas_ffn_bwd(const float* __restrict__ Y, const float* __restrict__ HPRE, const float* __restrict__ dOUT, const float* __restrict__ W1,
              const float* __restrict__ W2, const float* __restrict__ ln_gamma, float* __restrict__ HID, float* __restrict__ DHPRE,
              float* __restrict__ dY, float* __restrict__ g_gamma, float* __restrict__ g_beta, int64_t N) {
  constexpr int SS = S * S;
  __shared__ __align__(16) float sw[2 * SS + S];
  __shared__ float red[4 * 2 * S];
  for (int i = threadIdx.x; i < SS; i += blockDim.x) { sw[i] = W1[i]; sw[SS + i] = W2[i]; }
  if (threadIdx.x < S) sw[2 * SS + threadIdx.x] = ln_gamma[threadIdx.x];
  __syncthreads();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float dg[S], db[S];
#pragma unroll
  for (int i = 0; i < S; ++i) { dg[i] = 0.f; db[i] = 0.f; }
  if (n < N) {
    float y[S], h[S], g[S], dh[S], df[S];
    sas_load(dOUT + n * S, g);
    sas_load(HPRE + n * S, h);
    sas_matvec_t(g, sw + SS, dh);
#pragma unroll
    for (int i = 0; i < S; ++i) { dh[i] = h[i] > 0.f ? dh[i] : 0.f; h[i] = fmaxf(h[i], 0.f); }
    sas_store(HID + n * S, h);
    sas_store(DHPRE + n * S, dh);
    sas_matvec_t(dh, sw, df);
#pragma unroll
    for (int i = 0; i < S; ++i) df[i] += g[i];
    sas_load(Y + n * S, y);
    float mean = 0.f;
#pragma unroll
    for (int i = 0; i < S; ++i) mean += y[i];
    mean *= (1.0f / S);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < S; ++i) { const float d = y[i] - mean; var = fmaf(d, d, var); }
    var *= (1.0f / S);
    const float rstd = 1.0f / sqrtf(var + kLnEps);
    float xh[S];
#pragma unroll
    for (int i = 0; i < S; ++i) { xh[i] = (y[i] - mean) * rstd; dg[i] = df[i] * xh[i]; db[i] = df[i]; }
    sas_ln_bwd(df, xh, sw + 2 * SS, rstd, g);
    sas_store(dY + n * S, g);
  }
  sas_reduce_ln_grads(dg, db, g_gamma, g_beta, red);
}
void launch_sas_ffn_bwd(const float* Y, const float* HPRE, const float* dOUT, const float* W1, const float* W2, const float* ln_gamma,
                        float* HID, float* DHPRE, float* dY, float* g_gamma, float* g_beta, int64_t N, int S, cudaStream_t st) {
  PAMREC_PROF("sas_ffn_bwd", 1, st);
  if (N == 0) return;
  sas_widths(S, [&](auto w) {
    k_sas_ffn_bwd<decltype(w)::value><<<(unsigned)((N + 127) / 128), 128, 0, st>>>(Y, HPRE, dOUT, W1, W2, ln_gamma, HID, DHPRE, dY, g_gamma,
                                                                                   g_beta, N);
  });
}

// ------------------------------------------------------------------------------------------ read-out
// final_state = seq[b, length - 1] (zeros for a row without any satisfied item: tf.gather_nd on the GPU answers an index of -1 with
// zeros, oracle/siblings_oracle.py:sasrec_forward); U = final_state | target   (sasrec.py:72-78, 52-54)
template <int S>
__global__ void k_sas_final_fwd(const float* __restrict__ SEQ, const int* __restrict__ mask, const float* __restrict__ tgt,
                                float* __restrict__ U, int B, int T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 2 * S) return;
  const int b = i / (2 * S), j = i % (2 * S);
  if (j >= S) { U[i] = tgt[(int64_t)b * S + (j - S)]; return; }
  int len = 0;
  for (int t = 0; t < T; ++t) len += mask[(int64_t)b * T + t] == 1 ? 1 : 0;
  U[i] = len > 0 ? SEQ[((int64_t)b * T + (len - 1)) * S + j] : 0.f;
}
void launch_sas_final_fwd(const float* SEQ, const int* mask, const float* tgt, float* U, int B, int T, int S, cudaStream_t st) {
  PAMREC_PROF("sas_final_fwd", 1, st);
  if (B == 0) return;
  sas_widths(S, [&](auto w) {
    constexpr int S_ = decltype(w)::value;
    k_sas_final_fwd<S_><<<(B * 2 * S_ + 255) / 256, 256, 0, st>>>(SEQ, mask, tgt, U, B, T);
  });
}
// dSEQ = 0 except row length - 1 of every sample (dSEQ is zeroed by the caller); dTgt = dU[:, S:2S]
template <int S>
__global__ void k_sas_final_bwd(const float* __restrict__ dU, const int* __restrict__ mask, float* __restrict__ dSEQ, float* __restrict__ dTgt,
                                int B, int T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 2 * S) return;
  const int b = i / (2 * S), j = i % (2 * S);
  if (j >= S) { dTgt[(int64_t)b * S + (j - S)] = dU[i]; return; }
  int len = 0;
  for (int t = 0; t < T; ++t) len += mask[(int64_t)b * T + t] == 1 ? 1 : 0;
  if (len > 0) dSEQ[((int64_t)b * T + (len - 1)) * S + j] = dU[i];
}
void launch_sas_final_bwd(const float* dU, const int* mask, float* dSEQ, float* dTgt, int B, int T, int S, cudaStream_t st) {
  PAMREC_PROF("sas_final_bwd", 1, st);
  if (B == 0) return;
  cudaMemsetAsync(dSEQ, 0, (size_t)B * T * S * sizeof(float), st);
  sas_widths(S, [&](auto w) {
    constexpr int S_ = decltype(w)::value;
    k_sas_final_bwd<S_><<<(B * 2 * S_ + 255) / 256, 256, 0, st>>>(dU, mask, dSEQ, dTgt, B, T);
  });
}

// position table (one lookup row per (sample, position), sasrec.py:39-44): dPos[t] = sum_b dX0[b, t];  normsq += |dX0|^2 (the clip
// norm of an IndexedSlices gradient is taken over its un-deduplicated rows).  TS = T * S floats per sample.
__global__ void __launch_bounds__(128) k_sas_pos_bwd(const float* __restrict__ dX0, float* __restrict__ dPos, double* __restrict__ normsq,
                                                     int B, int TS) {
  __shared__ double sh[4];
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int b0 = blockIdx.y * 64, b1 = min(B, b0 + 64);
  float s = 0.f;
  double sq = 0.0;
  if (e < TS) {
    for (int b = b0; b < b1; ++b) { const float v = dX0[(int64_t)b * TS + e]; s += v; sq += (double)v * (double)v; }
    atomicAdd(dPos + e, s);
  }
  sq = warp_sum_d(sq);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = sq;
  __syncthreads();
  if (threadIdx.x == 0) { const double t = sh[0] + sh[1] + sh[2] + sh[3]; if (t != 0.0) atomicAdd(normsq, t); }
}
void launch_sas_pos_bwd(const float* dX0, float* dPos, double* normsq, int B, int T, int S, cudaStream_t st) { PAMREC_PROF("sas_pos_bwd", 1, st);
  if (B == 0) return;
  dim3 grid((T * S + 127) / 128, (B + 63) / 64);
  k_sas_pos_bwd<<<grid, 128, 0, st>>>(dX0, dPos, normsq, B, T * S);
}

}  // namespace pamrec
