// Kernels of the sibling multi-task baselines (SURVEY.md section 8(f) row N3): MMoEModel_original (models/sequential/mmoe.py),
// PLEModel (ple.py), ShareBottomModel (sharebottom.py).  What differs from PAMRec is the front end - two DIN-style attention
// poolings (`_attention_fcn`, mmoe.py:299-337) instead of the time-aware encoder - and the mixing layer; every dense layer,
// batch norm, the clip / Adam step and the sparse backward reuse the kernels of kernels_head.cu / kernels_optim.cu.
//
// Branch 0 = long_term (satisfied-only history, mmoe.py:199-207), branch 1 = short_term (full history, mmoe.py:208-216).
// Arrays indexed [2][N][.] use the ACTUAL token count N = B * T of the batch as the branch stride, so that the lookups of one
// table are one contiguous key list for the sparse plan.
#include "head_tiles.cuh"

namespace pamrec {

// The two width sets of the sibling models: (item, cate) = (16, 4) (config/mmoe.yaml) or (32, 8) (the reference's ple.yaml,
// sharebottom.yaml); a history token is E = item + cate floats.  Every kernel below is a template on <I, C>; the launchers pick the
// instantiation once per launch from the item width (pamrec_create admits no other pair).
template <int I_, int C_> struct SibW { static constexpr int I = I_, C = C_; };
template <typename F> static void sib_widths(int item_dim, F f) {
  if (item_dim == 32) f(SibW<32, 8>{});
  else f(SibW<16, 4>{});
}

// ------------------------------------------------------------------------------------------
// gather: h[r][n] = item_w[id] | cate_w[cid] for both histories, tgt[b] = item_w[item] | cate_w[cate]; the ids are copied into
// branch order for the sparse plan.  One thread per 16-byte chunk (E / 4 per token).
template <int I, int C>
__global__ void __launch_bounds__(256)
k_sib_gather(const int* __restrict__ sat_item, const int* __restrict__ sat_cate, const int* __restrict__ hist_item,
             const int* __restrict__ hist_cate, const int* __restrict__ items, const int* __restrict__ cates,
             const float* __restrict__ item_w, const float* __restrict__ cate_w, float* __restrict__ h, float* __restrict__ tgt,
             int* __restrict__ ids_item, int* __restrict__ ids_cate, int64_t N, int B) {
  constexpr int E = I + C, CH = E / 4, CI = I / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_hist = 2 * N * CH;
  if (i < n_hist) {
    const int64_t tok = i / CH;               // r * N + n
    const int c = (int)(i % CH);
    const int r = tok >= N ? 1 : 0;
    const int64_t n = tok - (int64_t)r * N;
    const int id = r == 0 ? sat_item[n] : hist_item[n];
    const int cid = r == 0 ? sat_cate[n] : hist_cate[n];
    if (c == 0) { if (ids_item) ids_item[tok] = id; if (ids_cate) ids_cate[tok] = cid; }
    const float4 v = c < CI ? ld4(item_w + (int64_t)id * I + 4 * c) : ld4(cate_w + (int64_t)cid * C + 4 * (c - CI));
    st4(h + tok * E + 4 * c, v);
  } else if (i < n_hist + (int64_t)B * CH) {
    const int64_t j = i - n_hist;
    const int b = (int)(j / CH), c = (int)(j % CH);
    const float4 v = c < CI ? ld4(item_w + (int64_t)items[b] * I + 4 * c) : ld4(cate_w + (int64_t)cates[b] * C + 4 * (c - CI));
    st4(tgt + (int64_t)b * E + 4 * c, v);
  }
}
void launch_sib_gather(const int* sat_item, const int* sat_cate, const int* hist_item, const int* hist_cate, const int* items,
                       const int* cates, const float* item_w, const float* cate_w, float* h, float* tgt, int* ids_item,
                       int* ids_cate, int B, int T, int item_dim, cudaStream_t st) { PAMREC_PROF("sib_gather", 1, st);
  if (B == 0) return;
  sib_widths(item_dim, [&](auto w) {
    constexpr int I = decltype(w)::I, C = decltype(w)::C, CH = (I + C) / 4;
    const int64_t N = (int64_t)B * T, total = 2 * N * CH + (int64_t)B * CH;
    k_sib_gather<I, C><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(sat_item, sat_cate, hist_item, hist_cate, items, cates, item_w,
                                                                         cate_w, h, tgt, ids_item, ids_cate, N, B);
  });
}

// has0[t] = 1 when id 0 is among the full-history or target ids of table t (0 item, 1 category): the rows that carry the L2
// term are tf.unique(history ids, target ids) (sequential_base_model.py:640-664); the satisfied-only history is a subset of the
// history EXCEPT for its padding id 0, so row 0 may be looked up (and receive a gradient) without being an L2 row.
__global__ void k_sib_has0(const int* __restrict__ hist_item, const int* __restrict__ hist_cate, const int* __restrict__ items,
                           const int* __restrict__ cates, int64_t N, int B, int* __restrict__ has0) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) {
    if (hist_item[i] == 0) has0[0] = 1;
    if (hist_cate[i] == 0) has0[1] = 1;
  } else if (i < N + B) {
    if (items[i - N] == 0) has0[0] = 1;
    if (cates[i - N] == 0) has0[1] = 1;
  }
}
void launch_sib_has0(const int* hist_item, const int* hist_cate, const int* items, const int* cates, int B, int T, int* has0,
                     cudaStream_t st) { PAMREC_PROF("sib_has0", 1, st);
  cudaMemsetAsync(has0, 0, 4 * sizeof(int), st);
  if (B == 0) return;
  const int64_t N = (int64_t)B * T;
  k_sib_has0<<<(unsigned)((N + B + 255) / 256), 256, 0, st>>>(hist_item, hist_cate, items, cates, N, B, has0);
}

// ------------------------------------------------------------------------------------------
// feature row of the attention MLP (mmoe.py:320-326): a = h A is already in feat[n, 4E r + 0:E]; fill q | a - q | a * q
template <int I, int C>
__global__ void __launch_bounds__(256) k_sib_feat_fwd(float* __restrict__ feat, const float* __restrict__ tgt, int64_t N, int T) {
  constexpr int E = I + C;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * 2 * E) return;
  const int64_t n = i / (2 * E);
  const int r = (int)((i % (2 * E)) / E), j = (int)(i % E);
  const int64_t b = n / T;
  float* f = feat + n * 8 * E + r * 4 * E;
  const float a = f[j], q = tgt[b * E + j];
  f[E + j] = q;
  f[2 * E + j] = a - q;
  f[3 * E + j] = a * q;
}
void launch_sib_feat_fwd(float* feat, const float* tgt, int B, int T, int item_dim, cudaStream_t st) { PAMREC_PROF("sib_feat_fwd", 1, st);
  if (B == 0) return;
  sib_widths(item_dim, [&](auto w) {
    constexpr int I = decltype(w)::I, C = decltype(w)::C;
    const int64_t N = (int64_t)B * T;
    k_sib_feat_fwd<I, C><<<(unsigned)((N * 2 * (I + C) + 255) / 256), 256, 0, st>>>(feat, tgt, N, T);
  });
}

// gradient of the feature row: d_a = df[0:E] + df[2E:3E] + df[3E:4E] * q  (-> d_att[r][n]);
// d_q[b][r] = sum_t df[E:2E] - df[2E:3E] + df[3E:4E] * a.   CTA = (sample, branch), thread = (t mod RY, feature), RY = 128 / E.
template <int I, int C>
__global__ void __launch_bounds__(128)
k_sib_feat_bwd(const float* __restrict__ d_feat, const float* __restrict__ feat, const float* __restrict__ tgt,
               float* __restrict__ d_att, float* __restrict__ dq, int64_t N, int T) {
  constexpr int E = I + C, RY = 128 / E;
  __shared__ float red[RY][E];
  const int b = blockIdx.x, r = blockIdx.y, tid = threadIdx.x;
  const int ty = tid / E, j = tid % E;
  float acc = 0.f;
  if (tid < RY * E) {
    const float q = tgt[(int64_t)b * E + j];
    for (int t = ty; t < T; t += RY) {
      const int64_t n = (int64_t)b * T + t;
      const float* df = d_feat + n * 8 * E + r * 4 * E;
      const float a = feat[n * 8 * E + r * 4 * E + j];
      const float d3 = df[3 * E + j], d2 = df[2 * E + j];
      d_att[((int64_t)r * N + n) * E + j] = df[j] + d2 + d3 * q;
      acc += df[E + j] - d2 + d3 * a;
    }
    red[ty][j] = acc;
  }
  __syncthreads();
  if (tid < E) {
    float s = 0.f;
#pragma unroll
    for (int y = 0; y < RY; ++y) s += red[y][tid];
    dq[((int64_t)b * 2 + r) * E + tid] = s;
  }
}
void launch_sib_feat_bwd(const float* d_feat, const float* feat, const float* tgt, float* d_att, float* dq, int B, int T, int item_dim,
                         cudaStream_t st) { PAMREC_PROF("sib_feat_bwd", 1, st);
  if (B == 0) return;
  sib_widths(item_dim, [&](auto w) {
    k_sib_feat_bwd<decltype(w)::I, decltype(w)::C><<<dim3(B, 2), 128, 0, st>>>(d_feat, feat, tgt, d_att, dq, (int64_t)B * T, T);
  });
}

// ------------------------------------------------------------------------------------------
// masked softmax over the history + weighted sum (mmoe.py:330-337, then reduce_sum over the sequence, mmoe.py:205-216):
// w = softmax_t(mask == 1 ? score : -(2^32)+1);  x[b, E r + j] = sum_t w_t h[r][b,t,j];  x[b, 2E:3E] = target.  Warp = (b, r).
__device__ __forceinline__ void sib_weights(const float* __restrict__ score, const int* __restrict__ mask, int64_t base, int T, int r,
                                            int lane, float* aw) {
  float s[8];
  float m = -INFINITY;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    float val = -INFINITY;
    if (t < T) val = (mask[base + t] == 1) ? score[(base + t) * 2 + r] : kMaskNeg;
    s[jj] = val;
    m = fmaxf(m, val);
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    const float e = (t < T) ? expf(s[jj] - m) : 0.f;
    s[jj] = e;
    sum += e;
  }
  sum = warp_sum(sum);
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    if (t < T) aw[t] = s[jj] / sum;
  }
  __syncwarp();
}

// lanes 0..19 own E / 20 adjacent columns each (one at E = 20, two at E = 40)
template <int I, int C>
__global__ void __launch_bounds__(128)
k_sib_pool_fwd(const float* __restrict__ h, const float* __restrict__ score, const int* __restrict__ sat_mask,
               const int* __restrict__ mask, const float* __restrict__ tgt, float* __restrict__ aw_out, float* __restrict__ x,
               int B, int T) {
  constexpr int E = I + C, CPL = E / 20;
  __shared__ float aws[4][PAMREC_MAX_T];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * 4 + w;
  if (unit >= 2 * B) return;
  const int b = unit >> 1, r = unit & 1;
  const int64_t N = (int64_t)B * T, base = (int64_t)b * T;
  float* aw = aws[w];
  sib_weights(score, r == 0 ? sat_mask : mask, base, T, r, lane, aw);
  for (int t = lane; t < T; t += 32) aw_out[(int64_t)r * N + base + t] = aw[t];
  if (lane < 20) {
    const int j0 = CPL * lane;
    const float* hr = h + ((int64_t)r * N + base) * E + j0;
    float acc[CPL];
#pragma unroll
    for (int k = 0; k < CPL; ++k) acc[k] = 0.f;
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int k = 0; k < CPL; ++k) acc[k] = fmaf(aw[t], hr[(int64_t)t * E + k], acc[k]);
    }
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      x[(int64_t)b * 3 * E + r * E + j0 + k] = acc[k];
      if (r == 0) x[(int64_t)b * 3 * E + 2 * E + j0 + k] = tgt[(int64_t)b * E + j0 + k];
    }
  }
}
void launch_sib_pool_fwd(const float* h, const float* score, const int* sat_mask, const int* mask, const float* tgt, float* aw,
                         float* x, int B, int T, int item_dim, cudaStream_t st) { PAMREC_PROF("sib_pool_fwd", 1, st);
  if (B == 0) return;
  sib_widths(item_dim, [&](auto w) {
    k_sib_pool_fwd<decltype(w)::I, decltype(w)::C><<<(2 * B + 3) / 4, 128, 0, st>>>(h, score, sat_mask, mask, tgt, aw, x, B, T);
  });
}

// backward: d_out = d_x[b, E r : E r + E];  dw_t = d_out . h_t;  d_score_t = mask ? w_t (dw_t - sum_s w_s dw_s) : 0;
// dh[r][n] = w_t d_out  (the attention_mat path is added afterwards by the dX GEMM of d_att)
template <int I, int C>
__global__ void __launch_bounds__(128)
k_sib_pool_bwd(const float* __restrict__ h, const float* __restrict__ aw_in, const int* __restrict__ sat_mask,
               const int* __restrict__ mask, const float* __restrict__ d_x, float* __restrict__ d_score, float* __restrict__ dh,
               int B, int T) {
  constexpr int E = I + C, CH = E / 4;
  __shared__ __align__(16) float dout[4][E];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * 4 + w;
  if (unit >= 2 * B) return;
  const int b = unit >> 1, r = unit & 1;
  const int64_t N = (int64_t)B * T, base = (int64_t)b * T;
  const int* mk = r == 0 ? sat_mask : mask;
  for (int j = lane; j < E; j += 32) dout[w][j] = d_x[(int64_t)b * 3 * E + r * E + j];
  __syncwarp();
  float4 d[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) d[c] = ld4(&dout[w][4 * c]);
  float dw[8], a[8];
  float dot = 0.f;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    float v = 0.f, at = 0.f;
    if (t < T) {
      const float* hr = h + ((int64_t)r * N + base + t) * E;
#pragma unroll
      for (int c = 0; c < CH; ++c) v += f4_dot(d[c], ld4(hr + 4 * c));
      at = aw_in[(int64_t)r * N + base + t];
      dot = fmaf(at, v, dot);
    }
    dw[jj] = v; a[jj] = at;
  }
  dot = warp_sum(dot);
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    if (t < T) {
      d_score[(base + t) * 2 + r] = (mk[base + t] == 1) ? a[jj] * (dw[jj] - dot) : 0.f;
      float* o = dh + ((int64_t)r * N + base + t) * E;
#pragma unroll
      for (int c = 0; c < CH; ++c) st4(o + 4 * c, make_float4(a[jj] * d[c].x, a[jj] * d[c].y, a[jj] * d[c].z, a[jj] * d[c].w));
    }
  }
}
void launch_sib_pool_bwd(const float* h, const float* aw, const int* sat_mask, const int* mask, const float* d_x, float* d_score,
                         float* dh, int B, int T, int item_dim, cudaStream_t st) { PAMREC_PROF("sib_pool_bwd", 1, st);
  if (B == 0) return;
  sib_widths(item_dim, [&](auto w) {
    k_sib_pool_bwd<decltype(w)::I, decltype(w)::C><<<(2 * B + 3) / 4, 128, 0, st>>>(h, aw, sat_mask, mask, d_x, d_score, dh, B, T);
  });
}

// gradient of the target rows: towers' target columns (d_tgt, MMoE / PLE) + x's target columns + the query of both branches
template <int I, int C>
__global__ void k_sib_tgt_total(const float* __restrict__ d_tgt, const float* __restrict__ d_x, const float* __restrict__ dq,
                                float* __restrict__ out, int B) {
  constexpr int E = I + C;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * E) return;
  const int b = i / E, j = i % E;
  float s = d_x[(int64_t)b * 3 * E + 2 * E + j] + dq[((int64_t)b * 2) * E + j] + dq[((int64_t)b * 2 + 1) * E + j];
  if (d_tgt != nullptr) s += d_tgt[i];
  out[i] = s;
}
void launch_sib_tgt_total(const float* d_tgt, const float* d_x, const float* dq, float* out, int B, int item_dim, cudaStream_t st) {
  PAMREC_PROF("sib_tgt_total", 1, st);
  if (B == 0) return;
  sib_widths(item_dim, [&](auto w) {
    constexpr int I = decltype(w)::I, C = decltype(w)::C;
    k_sib_tgt_total<I, C><<<(B * (I + C) + 255) / 256, 256, 0, st>>>(d_tgt, d_x, dq, out, B);
  });
}

// ------------------------------------------------------------------------------------------
// mixing (mmoe.py:43-50, ple.py:51-58): a gate is a BN + ReLU MLP like any other (no softmax);
// out_g = sum_j gate_g[j] * expert_{sel[g][j]};  U = main | tgt | sub | tgt  (two tower inputs of 64 + E)
struct MixSel { int s[2][5]; };
template <int I, int C>
__global__ void __launch_bounds__(64)
k_sib_mix_fwd(const float* __restrict__ ZE1, const float* __restrict__ ZG1, BnSet e1, BnSet g1, const float* __restrict__ tgt,
              float* __restrict__ U, int ldE, MixSel sel) {
  constexpr int E = I + C, TI = 64 + E;
  __shared__ float gt[10];
  const int b = blockIdx.x, c = threadIdx.x;
  if (c < 10) gt[c] = bn_relu(ZG1[(int64_t)b * 10 + c], g1.stat, g1.gamma, g1.beta, c);
  __syncthreads();
  float mn = 0.f, sb = 0.f;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int em = sel.s[0][j] * 64 + c, es = sel.s[1][j] * 64 + c;
    mn = fmaf(gt[j], bn_relu(ZE1[(int64_t)b * ldE + em], e1.stat, e1.gamma, e1.beta, em), mn);
    sb = fmaf(gt[5 + j], bn_relu(ZE1[(int64_t)b * ldE + es], e1.stat, e1.gamma, e1.beta, es), sb);
  }
  float* u = U + (int64_t)b * 2 * TI;
  u[c] = mn;
  u[TI + c] = sb;
  if (c < E) { const float t = tgt[(int64_t)b * E + c]; u[64 + c] = t; u[TI + 64 + c] = t; }
}
void launch_sib_mix_fwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* tgt, float* U, int n_expert,
                        const int sel[2][5], int B, int item_dim, cudaStream_t st) { PAMREC_PROF("sib_mix_fwd", 1, st);
  if (B == 0) return;
  MixSel s;
  for (int g = 0; g < 2; ++g) for (int j = 0; j < 5; ++j) s.s[g][j] = sel[g][j];
  sib_widths(item_dim, [&](auto w) {
    k_sib_mix_fwd<decltype(w)::I, decltype(w)::C><<<B, 64, 0, st>>>(ZE1, ZG1, e1, g1, tgt, U, n_expert * 64, s);
  });
}

// dE1[e] = sum over (gate g, slot j) with sel[g][j] == e of gate_g[j] * d_out_g;  dG1[g][j] = expert_{sel[g][j]} . d_out_g;
// dTgt = dU[64:64+E] + dU[TI+64:TI+64+E]
template <int I, int C>
__global__ void __launch_bounds__(64)
k_sib_mix_bwd(const float* __restrict__ ZE1, const float* __restrict__ ZG1, BnSet e1, BnSet g1, const float* __restrict__ dU,
              float* __restrict__ dE1, float* __restrict__ dG1, float* __restrict__ dTgt, int n_expert, MixSel sel) {
  constexpr int E = I + C, TI = 64 + E;
  __shared__ float gt[10];
  __shared__ float red[2][10];
  const int b = blockIdx.x, c = threadIdx.x, lane = c & 31, w = c >> 5;
  const int ldE = n_expert * 64;
  if (c < 10) gt[c] = bn_relu(ZG1[(int64_t)b * 10 + c], g1.stat, g1.gamma, g1.beta, c);
  __syncthreads();
  const float* du = dU + (int64_t)b * 2 * TI;
  const float dm = du[c], ds = du[TI + c];
  if (c < E) dTgt[(int64_t)b * E + c] = du[64 + c] + du[TI + 64 + c];
  for (int e = 0; e < n_expert; ++e) {
    float v = 0.f;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      if (sel.s[0][j] == e) v = fmaf(gt[j], dm, v);
      if (sel.s[1][j] == e) v = fmaf(gt[5 + j], ds, v);
    }
    dE1[(int64_t)b * ldE + e * 64 + c] = v;
  }
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int em = sel.s[0][j] * 64 + c, es = sel.s[1][j] * 64 + c;
    const float pm = warp_sum(bn_relu(ZE1[(int64_t)b * ldE + em], e1.stat, e1.gamma, e1.beta, em) * dm);
    const float ps = warp_sum(bn_relu(ZE1[(int64_t)b * ldE + es], e1.stat, e1.gamma, e1.beta, es) * ds);
    if (lane == 0) { red[w][j] = pm; red[w][5 + j] = ps; }
  }
  __syncthreads();
  if (c < 10) dG1[(int64_t)b * 10 + c] = red[0][c] + red[1][c];
}
void launch_sib_mix_bwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* dU, float* dE1, float* dG1,
                        float* dTgt, int n_expert, const int sel[2][5], int B, int item_dim, cudaStream_t st) {
  PAMREC_PROF("sib_mix_bwd", 1, st);
  if (B == 0) return;
  MixSel s;
  for (int g = 0; g < 2; ++g) for (int j = 0; j < 5; ++j) s.s[g][j] = sel[g][j];
  sib_widths(item_dim, [&](auto w) {
    k_sib_mix_bwd<decltype(w)::I, decltype(w)::C><<<B, 64, 0, st>>>(ZE1, ZG1, e1, g1, dU, dE1, dG1, dTgt, n_expert, s);
  });
}

// ------------------------------------------------------------------------------------------
// loss = mean xent(logit, labels) + aux_w * mean xent(valid_logit, labels_play)   (mmoe.py:52-82; aux_w is the literal 0.5)
__device__ __forceinline__ float sib_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float sib_xent(float x, float y) { return fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x))); }
__global__ void __launch_bounds__(1024)
k_sib_loss(const float* __restrict__ logits, const float* __restrict__ y_sat, const float* __restrict__ y_play,
           float* __restrict__ d_logits, double* __restrict__ loss_acc, int B, float aux_w, int heads) {
  __shared__ double sh[2][32];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const float inv_b = 1.0f / (float)B;
  double a0 = 0.0, a1 = 0.0;
  for (int b = tid; b < B; b += blockDim.x) {
    const float x0 = logits[heads * b], y0 = y_sat[b];
    a0 += (double)sib_xent(x0, y0);
    d_logits[heads * b] = (sib_sigmoid(x0) - y0) * inv_b;
    if (heads == 2) {
      const float x1 = logits[2 * b + 1], y1 = y_play[b];
      a1 += (double)sib_xent(x1, y1);
      d_logits[2 * b + 1] = aux_w * (sib_sigmoid(x1) - y1) * inv_b;
    }
  }
  a0 = warp_sum_d(a0); a1 = warp_sum_d(a1);
  if (lane == 0) { sh[0][w] = a0; sh[1][w] = a1; }
  __syncthreads();
  if (tid == 0) {
    double t0 = 0.0, t1 = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { t0 += sh[0][k]; t1 += sh[1][k]; }
    loss_acc[0] = t0 / (double)B;
    loss_acc[1] = (double)aux_w * t1 / (double)B;
    loss_acc[2] = 0.0;
  }
}
void launch_sib_loss(const float* logits, const float* y_sat, const float* y_play, float* d_logits, double* loss_acc, int B, float aux_w,
                     int heads, cudaStream_t st) { PAMREC_PROF("sib_loss", 1, st);
  k_sib_loss<<<1, 1024, 0, st>>>(logits, y_sat, y_play, d_logits, loss_acc, B, aux_w, heads);
}

__global__ void k_sib_pred(const float* __restrict__ logits, float* __restrict__ pred, int B, int heads) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) pred[b] = sib_sigmoid(logits[heads * b]);
}
void launch_sib_pred(const float* logits, float* pred, int B, int heads, cudaStream_t st) { PAMREC_PROF("sigmoid", 1, st);
  if (B == 0) return;
  k_sib_pred<<<(B + 255) / 256, 256, 0, st>>>(logits, pred, B, heads);
}

}  // namespace pamrec
