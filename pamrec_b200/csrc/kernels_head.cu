// Head kernels: grouped dense layers with batch-norm-on-load, batch-norm statistics
// (forward and backward), attention pooling, MMoE mixing and the fused three-term loss.
//
// Batch norm in the reference is the non-fused Keras path (pamrec.py:366-372,
// base_model.py:680-686): biased batch variance, eps 1e-4, momentum 0.95.  Every BN layer
// is a grid-wide reduction, so a layer is split as  [dense + column sums] -> [finalize] ->
// [next dense applies BN+ReLU while loading its input].  Sums are accumulated in fp64
// (atomics) so that var = E[z^2] - E[z]^2 does not lose digits.
#include "head_tiles.cuh"

namespace pamrec {

// ------------------------------------------------------------------------------------------
// Z[m, zo+n] = sum_k act(X[m, xo+k]) W_g[k][n] + b_g[n]   (+ fp64 column sums of Z for the next batch norm)
__global__ void __launch_bounds__(kHT) k_dense_fwd(const DenseP p, int tiles_m) {
  __shared__ __align__(16) unsigned char smem[kDenseFwdSmem];
  dense_fwd_item(p, p.M, p.out_sums, tiles_m, blockIdx.x, gridDim.x, blockIdx.y, smem);
}

void launch_dense_fwd(const DenseP& p, cudaStream_t st) { PAMREC_PROF("dense_fwd", 1, st);
  if (p.M == 0) return;
  const FwdGrid g = dense_fwd_grid(p.M, p.n_groups, p.N, 148 * 8);
  k_dense_fwd<<<dim3(g.gx, g.ny), kHT, 0, st>>>(p, g.tiles_m);
}

// ------------------------------------------------------------------------------------------
// dX[m, out_off[s]+k] (+)= sum over contributions c of slice s: sum_n dZ[m, dz_off+n] W_c[k][n]
__global__ void __launch_bounds__(kHT) k_dense_dx(const DenseDxP p) {
  __shared__ __align__(16) unsigned char smem[kDenseDxSmem];
  dense_dx_item(p, p.M, p.g.count, blockIdx.x, blockIdx.y, smem);
}

void launch_dense_dx(const DenseDxP& p, cudaStream_t st) { PAMREC_PROF("dense_dx", 1, st);
  if (p.M == 0) return;
  const DxGrid g = dense_dx_grid(p.M, p.n_slices, p.K);
  k_dense_dx<<<dim3(g.gx, g.ny), kHT, 0, st>>>(p);
}

// ------------------------------------------------------------------------------------------
// dW_g[k][n] += sum_m act(X[m, xo+k]) dZ[m, zo+n];  db_g[n] += sum_m dZ[m, zo+n].  The contraction runs over rows:
// a CTA takes `rows_per_cta` rows in sub-chunks of 32 and one 32 x 32 tile of (k, n); partial sums leave by atomicAdd.
__global__ void __launch_bounds__(kHT) k_dense_dw(const DenseDwP p, int rows_per_cta) {
  __shared__ __align__(16) unsigned char smem[kDenseDwSmem];
  dense_dw_item(p, p.M, p.g.count, rows_per_cta, blockIdx.x, blockIdx.y, smem);
}

void launch_dense_dw(const DenseDwP& p, cudaStream_t st) { PAMREC_PROF("dense_dw", 1, st);
  if (p.M == 0) return;
  const DwGrid g = dense_dw_grid(p.M, p.n_groups, p.K, p.N, 148 * 6);
  k_dense_dw<<<dim3(g.chunks, g.ny), kHT, 0, st>>>(p, g.rows_per_cta);
}

// ------------------------------------------------------------------------------------------
__global__ void k_bn_finalize(BnSet s, double count) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= s.C) return;
  double mean = s.sums[2 * c] / count;
  double var = s.sums[2 * c + 1] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  s.stat[2 * c] = (float)mean;
  s.stat[2 * c + 1] = (float)(1.0 / sqrt(var + (double)kBnEps));
  // assign_moving_average: variable -= (variable - value) * (1 - momentum)
  s.mmean[c] -= (s.mmean[c] - (float)mean) * kBnDecay;
  s.mvar[c] -= (s.mvar[c] - (float)var) * kBnDecay;
  s.sums[2 * c] = 0.0;
  s.sums[2 * c + 1] = 0.0;
}
void launch_bn_finalize(const BnSet& s, double count, cudaStream_t st) { PAMREC_PROF("bn_finalize", 1, st);
  k_bn_finalize<<<(s.C + 127) / 128, 128, 0, st>>>(s, count);
}
__global__ void k_bn_eval_stat(BnSet s) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= s.C) return;
  s.stat[2 * c] = s.mmean[c];
  s.stat[2 * c + 1] = 1.0f / sqrtf(s.mvar[c] + kBnEps);
}
void launch_bn_eval_stat(const BnSet& s, cudaStream_t st) { PAMREC_PROF("bn_eval_stat", 1, st); k_bn_eval_stat<<<(s.C + 127) / 128, 128, 0, st>>>(s); }

constexpr int kBnRowsPerThread = 8;
__global__ void __launch_bounds__(256) k_bn_bwd_stats(BnSet s, const float* __restrict__ dA, const float* __restrict__ Z, int M) {
  __shared__ double sh[2][256];
  const int cb = min(s.C, 32), rl = 256 / cb;
  const int tid = threadIdx.x, ry = tid / cb, cx = tid % cb;
  const int col = blockIdx.x * cb + cx;
  const int rpb = rl * kBnRowsPerThread;
  double s1 = 0.0, s2 = 0.0;
  if (ry < rl && col < s.C) {
    const float mean = s.stat[2 * col], inv = s.stat[2 * col + 1], g = s.gamma[col], be = s.beta[col];
    const int r0 = blockIdx.y * rpb + ry;
#pragma unroll
    for (int k = 0; k < kBnRowsPerThread; ++k) {
      int r = r0 + k * rl;
      if (r < M) {
        float xh = (Z[(int64_t)r * s.C + col] - mean) * inv;
        float y = fmaf(g, xh, be);
        float dy = y > 0.f ? dA[(int64_t)r * s.C + col] : 0.f;
        s1 += (double)dy;
        s2 += (double)dy * (double)xh;
      }
    }
  }
  sh[0][tid] = s1; sh[1][tid] = s2;
  __syncthreads();
  if (ry == 0 && col < s.C) {
    for (int k = 1; k < rl; ++k) { s1 += sh[0][k * cb + cx]; s2 += sh[1][k * cb + cx]; }
    atomicAdd(s.bsums + 2 * col, s1);
    atomicAdd(s.bsums + 2 * col + 1, s2);
  }
}
void launch_bn_bwd_stats(const BnSet& s, const float* dA, const float* Z, int M, cudaStream_t st) { PAMREC_PROF("bn_bwd_stats", 1, st);
  if (M == 0) return;
  int cb = s.C < 32 ? s.C : 32;
  int rpb = (256 / cb) * kBnRowsPerThread;
  dim3 grid((s.C + cb - 1) / cb, (M + rpb - 1) / rpb);
  k_bn_bwd_stats<<<grid, 256, 0, st>>>(s, dA, Z, M);
}

// ------------------------------------------------------------------------------------------
// P1 (pamrec.py:272-282): s = relu(BN(z2)); a = softmax_t(mask==1 ? s : -(2^32)+1); new_long = sum_t a_t h_t
// warp per sample.
__device__ __forceinline__ void pool_weights(const float* __restrict__ Z2, const BnSet& s1, const int* __restrict__ mask,
                                             int64_t base, int T, int lane, float* aw) {
  const float mean = s1.stat[0], inv = s1.stat[1], g = s1.gamma[0], be = s1.beta[0];
  float s[8];
  float m = -INFINITY;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    int t = jj * 32 + lane;
    float val = -INFINITY;
    if (t < T) {
      float sv = fmaxf(fmaf(g, (Z2[base + t] - mean) * inv, be), 0.f);
      val = (mask[base + t] == 1) ? sv : kMaskNeg;
    }
    s[jj] = val;
    m = fmaxf(m, val);
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    int t = jj * 32 + lane;
    float e = (t < T) ? expf(s[jj] - m) : 0.f;
    s[jj] = e;
    sum += e;
  }
  sum = warp_sum(sum);
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    int t = jj * 32 + lane;
    if (t < T) aw[t] = s[jj] / sum;
  }
  __syncwarp();
}

__global__ void __launch_bounds__(128) k_pool_fwd(const float* __restrict__ H, const float* __restrict__ Z2, BnSet s1,
                                                  const int* __restrict__ mask, float* __restrict__ new_long, float* __restrict__ aw_out,
                                                  int B, int T) {
  __shared__ float aws[4][PAMREC_MAX_T];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 4 + w;
  if (b >= B) return;
  const int64_t base = (int64_t)b * T;
  float* aw = aws[w];
  pool_weights(Z2, s1, mask, base, T, lane, aw);
  if (aw_out) for (int t = lane; t < T; t += 32) aw_out[base + t] = aw[t];
  const int tg = lane / 10, c = lane % 10;
  float4 acc = f4_zero();
  if (lane < 30)
    for (int t = tg; t < T; t += 3) f4_fma(acc, aw[t], ld4(H + (base + t) * kD + 4 * c));
  float4 a1 = f4_shfl_down(acc, 10), a2 = f4_shfl_down(acc, 20);
  if (lane < 10) {
    acc.x += a1.x + a2.x; acc.y += a1.y + a2.y; acc.z += a1.z + a2.z; acc.w += a1.w + a2.w;
    st4(new_long + (int64_t)b * kD + 4 * c, acc);
  }
}
void launch_pool_fwd(const float* H, const float* Z2, const BnSet& s1, const int* mask, float* new_long, float* aw_out, int B, int T,
                     cudaStream_t st) { PAMREC_PROF("pool_fwd", 1, st);
  if (B == 0) return;
  k_pool_fwd<<<(B + 3) / 4, 128, 0, st>>>(H, Z2, s1, mask, new_long, aw_out, B, T);
}

// backward of the pooling: dA2[b,t] = grad wrt s_t (post-ReLU score), dH[b,t,:] = a_t * d_new_long[b,:]
__global__ void __launch_bounds__(128) k_pool_bwd(const float* __restrict__ H, const float* __restrict__ Z2, BnSet s1,
                                                  const int* __restrict__ mask, const float* __restrict__ dNL,
                                                  float* __restrict__ dA2, float* __restrict__ dH, int B, int T) {
  __shared__ float aws[4][PAMREC_MAX_T];
  __shared__ __align__(16) float dnls[4][kD];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 4 + w;
  if (b >= B) return;
  const int64_t base = (int64_t)b * T;
  float* aw = aws[w];
  pool_weights(Z2, s1, mask, base, T, lane, aw);
  for (int i = lane; i < kD; i += 32) dnls[w][i] = dNL[(int64_t)b * kD + i];
  __syncwarp();
  float4 dn[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) dn[i] = ld4(&dnls[w][4 * i]);
  float da[8];
  float dot = 0.f;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    int t = jj * 32 + lane;
    float v = 0.f;
    if (t < T) {
      const float* h = H + (base + t) * kD;
#pragma unroll
      for (int i = 0; i < 10; ++i) v += f4_dot(dn[i], ld4(h + 4 * i));
      dot = fmaf(aw[t], v, dot);
    }
    da[jj] = v;
  }
  dot = warp_sum(dot);
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    int t = jj * 32 + lane;
    if (t < T) dA2[base + t] = (mask[base + t] == 1) ? aw[t] * (da[jj] - dot) : 0.f;
  }
  const int tg = lane / 10, c = lane % 10;
  if (lane < 30)
    for (int t = tg; t < T; t += 3) {
      float a = aw[t];
      float4 d = ld4(&dnls[w][4 * c]);   // dn[c] with a runtime c would spill: re-read the chunk from smem
      st4(dH + (base + t) * kD + 4 * c, make_float4(a * d.x, a * d.y, a * d.z, a * d.w));
    }
}
void launch_pool_bwd(const float* H, const float* Z2, const BnSet& s1, const int* mask, const float* dNL, float* dA2,
                     float* dH, int B, int T, cudaStream_t st) { PAMREC_PROF("pool_bwd", 1, st);
  if (B == 0) return;
  k_pool_bwd<<<(B + 3) / 4, 128, 0, st>>>(H, Z2, s1, mask, dNL, dA2, dH, B, T);
}

// ------------------------------------------------------------------------------------------
// M1 mixing (pamrec.py:46-50, 315-316): main = sum_j gate_main[j] e_j ; U = main|tgt|sub|tgt
__global__ void __launch_bounds__(64) k_combine_fwd(const float* __restrict__ ZE1, const float* __restrict__ ZG1, BnSet e1,
                                                    BnSet g1, const float* __restrict__ tgt, float* __restrict__ U, int B) {
  __shared__ float gt[10];
  const int b = blockIdx.x, c = threadIdx.x;
  if (c < 10) gt[c] = bn_relu(ZG1[(int64_t)b * 10 + c], g1.stat, g1.gamma, g1.beta, c);
  __syncthreads();
  float mn = 0.f, sb = 0.f;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    float e = bn_relu(ZE1[(int64_t)b * 320 + j * 64 + c], e1.stat, e1.gamma, e1.beta, j * 64 + c);
    mn = fmaf(gt[j], e, mn);
    sb = fmaf(gt[5 + j], e, sb);
  }
  float* u = U + (int64_t)b * 168;
  u[c] = mn;
  u[84 + c] = sb;
  if (c < kE) { float t = tgt[(int64_t)b * kE + c]; u[64 + c] = t; u[148 + c] = t; }
}
void launch_combine_fwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* tgt, float* U,
                        int B, cudaStream_t st) { PAMREC_PROF("combine_fwd", 1, st);
  if (B == 0) return;
  k_combine_fwd<<<B, 64, 0, st>>>(ZE1, ZG1, e1, g1, tgt, U, B);
}

__global__ void __launch_bounds__(64) k_combine_bwd(const float* __restrict__ ZE1, const float* __restrict__ ZG1, BnSet e1,
                                                    BnSet g1, const float* __restrict__ dU, float* __restrict__ dE1,
                                                    float* __restrict__ dG1, float* __restrict__ dTgt, int B) {
  __shared__ float gt[10];
  __shared__ float red[2][10];
  const int b = blockIdx.x, c = threadIdx.x, lane = c & 31, w = c >> 5;
  if (c < 10) gt[c] = bn_relu(ZG1[(int64_t)b * 10 + c], g1.stat, g1.gamma, g1.beta, c);
  __syncthreads();
  const float* du = dU + (int64_t)b * 168;
  const float dm = du[c], ds = du[84 + c];
  if (c < kE) dTgt[(int64_t)b * kE + c] = du[64 + c] + du[148 + c];
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    float e = bn_relu(ZE1[(int64_t)b * 320 + j * 64 + c], e1.stat, e1.gamma, e1.beta, j * 64 + c);
    dE1[(int64_t)b * 320 + j * 64 + c] = gt[j] * dm + gt[5 + j] * ds;
    float pm = warp_sum(e * dm), ps = warp_sum(e * ds);
    if (lane == 0) { red[w][j] = pm; red[w][5 + j] = ps; }
  }
  __syncthreads();
  if (c < 10) dG1[(int64_t)b * 10 + c] = red[0][c] + red[1][c];
}
void launch_combine_bwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* dU, float* dE1,
                        float* dG1, float* dTgt, int B, cudaStream_t st) { PAMREC_PROF("combine_bwd", 1, st);
  if (B == 0) return;
  k_combine_bwd<<<B, 64, 0, st>>>(ZE1, ZG1, e1, g1, dU, dE1, dG1, dTgt, B);
}

// ------------------------------------------------------------------------------------------
// L1 + L2 + L3 and their gradients in one kernel (base_model.py:196-205, pamrec.py:70-106).
// ApproxNDCG restated from TensorFlow-Ranking 0.3.x (see oracle/pamrec_oracle.py:approx_ndcg_loss).
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float xent_(float x, float y) { return fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x))); }

__device__ double block_sum_d(double v, double* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum_d(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = (lane < (int)(blockDim.x >> 5)) ? sh[lane] : 0.0;
    r = warp_sum_d(r);
    if (lane == 0) sh[0] = r;
  }
  __syncthreads();
  r = sh[0];
  return r;
}

__global__ void __launch_bounds__(1024)
k_loss(const float* __restrict__ logits, const float* __restrict__ y_sat, const float* __restrict__ y_play,
       const float* __restrict__ plays, float* __restrict__ d_logits, double* __restrict__ loss_acc, int B, int B_global,
       const double* __restrict__ n_valid_global, float fuzhu_w, float order_w, int sm_group) {
  __shared__ double sh[32];
  const int tid = threadIdx.x;
  const int G = B / PAMREC_GROUP;
  double cnt = 0.0;
  for (int g = tid; g < G; g += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < PAMREC_GROUP; ++i) s += plays[g * PAMREC_GROUP + i];
    cnt += (s > 0.f) ? 1.0 : 0.0;
  }
  double nval_local = block_sum_d(cnt, sh);
  const double nval = n_valid_global ? *n_valid_global : nval_local;   // data parallel: count over all ranks
  const float inv_b = 1.0f / (float)B_global;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0;
  if (sm_group == 0) {
    for (int b = tid; b < B; b += blockDim.x) {
      float x0 = logits[3 * b], x1 = logits[3 * b + 1];
      float y0 = y_sat[b], y1 = y_play[b];
      a0 += (double)xent_(x0, y0);
      a1 += (double)xent_(x1, y1);
      d_logits[3 * b] = (sigmoidf_(x0) - y0) * inv_b;
      d_logits[3 * b + 1] = fuzhu_w * (sigmoidf_(x1) - y1) * inv_b;
    }
  } else {
    // hparams.loss == "softmax" (base_model.py:222-242, pamrec.py:97-105):  -group * mean(log(where(y == 1, softmax, 1))) over all
    // B elements = -(group / B) * sum over positives of log softmax;  d/dx_j = (group / B) * (n_pos * softmax_j - [y_j == 1])
    const float scale = (float)sm_group * inv_b;
    for (int u = tid; u < 2 * (B / sm_group); u += blockDim.x) {
      const int head = u & 1, r0 = (u >> 1) * sm_group;
      const float* y = head ? y_play : y_sat;
      float mx = -INFINITY;
      for (int i = 0; i < sm_group; ++i) mx = fmaxf(mx, logits[3 * (r0 + i) + head]);
      float se = 0.f;
      int n_pos = 0;
      for (int i = 0; i < sm_group; ++i) { se += expf(logits[3 * (r0 + i) + head] - mx); n_pos += y[r0 + i] == 1.0f; }
      const float lse = mx + logf(se), w = head ? fuzhu_w : 1.0f;
      double acc = 0.0;
      for (int i = 0; i < sm_group; ++i) {
        const float x = logits[3 * (r0 + i) + head];
        const bool pos = y[r0 + i] == 1.0f;
        if (pos) acc += (double)(lse - x);
        d_logits[3 * (r0 + i) + head] = w * scale * ((float)n_pos * expf(x - lse) - (pos ? 1.0f : 0.f));
      }
      if (head) a1 += acc * (double)sm_group; else a0 += acc * (double)sm_group;
    }
  }
  const float alpha = 10.0f;
  for (int g = tid; g < G; g += blockDim.x) {
    float o[5], s[5], y[5], gain[5], rank[5], dLr[5];
    float lsum = 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      o[i] = logits[3 * (g * 5 + i) + 2];
      s[i] = sigmoidf_(o[i]);                      // pamrec.py:74
      y[i] = plays[g * 5 + i];
      lsum += y[i];
    }
    const bool valid = lsum > 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      float yy = valid ? y[i] : 1e-10f;
      y[i] = yy;
      gain[i] = exp2f(yy) - 1.0f;
    }
    float dcg = 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      float r = 0.5f;
#pragma unroll
      for (int j = 0; j < 5; ++j) r += sigmoidf_(alpha * (s[j] - s[i]));
      rank[i] = r;
      dcg += gain[i] / log1pf(r);
    }
    float ys[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) ys[i] = y[i];
#pragma unroll
    for (int i = 0; i < 4; ++i)                    // sort descending (5 elements)
#pragma unroll
      for (int j = 0; j < 4 - i; ++j)
        if (ys[j] < ys[j + 1]) { float tmp = ys[j]; ys[j] = ys[j + 1]; ys[j + 1] = tmp; }
    float idcg = 0.f;
#pragma unroll
    for (int r = 0; r < 5; ++r) idcg += (exp2f(ys[r]) - 1.0f) / log1pf((float)(r + 1));
    const float inv = idcg > 0.f ? 1.0f / idcg : 0.f;
    const float w = valid ? 1.0f : 0.f;
    a2 += (double)(w * -(dcg * inv));
    const float coef = (nval > 0.0) ? order_w * w / (float)nval : 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      float l1p = log1pf(rank[i]);
      dLr[i] = gain[i] * inv / (l1p * l1p * (1.0f + rank[i]));
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        if (i == j) continue;
        float sij = sigmoidf_(alpha * (s[j] - s[i]));   // d rank_i / d s_j
        float sji = sigmoidf_(alpha * (s[i] - s[j]));   // d rank_j / d s_j (negative sign)
        acc += dLr[i] * alpha * sij * (1.0f - sij) - dLr[j] * alpha * sji * (1.0f - sji);
      }
      d_logits[3 * (g * 5 + j) + 2] = coef * acc * s[j] * (1.0f - s[j]);
    }
  }
  for (int b = G * 5 + tid; b < B; b += blockDim.x) d_logits[3 * b + 2] = 0.f;
  a0 = block_sum_d(a0, sh);
  a1 = block_sum_d(a1, sh);
  a2 = block_sum_d(a2, sh);
  if (tid == 0) {
    loss_acc[0] = a0 / (double)B_global;
    loss_acc[1] = (double)fuzhu_w * a1 / (double)B_global;
    loss_acc[2] = nval > 0.0 ? (double)order_w * a2 / nval : 0.0;
  }
}
void launch_loss(const float* logits, const float* y_sat, const float* y_play, const float* plays, float* d_logits,
                 double* loss_acc, int B, int B_global, const double* n_valid_global, float fuzhu_w, float order_w,
                 int softmax_group, cudaStream_t st) { PAMREC_PROF("loss", 1, st);
  k_loss<<<1, 1024, 0, st>>>(logits, y_sat, y_play, plays, d_logits, loss_acc, B, B_global, n_valid_global, fuzhu_w, order_w,
                             softmax_group);
}

__global__ void k_sigmoid_col0(const float* __restrict__ logits, float* __restrict__ pred, int B) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) pred[b] = sigmoidf_(logits[3 * b]);
}
void launch_sigmoid_col0(const float* logits, float* pred, int B, cudaStream_t st) { PAMREC_PROF("sigmoid", 1, st);
  if (B == 0) return;
  k_sigmoid_col0<<<(B + 255) / 256, 256, 0, st>>>(logits, pred, B);
}

}  // namespace pamrec
