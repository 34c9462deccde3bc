// Tile bodies of the stand-alone head kernels (kernels_head.cu, the PAMREC_HEAD_LEGACY=1 / no-cooperative-launch path) as
// device functions: one "item" = what one CTA of kHT threads does, called with (blockIdx, gridDim).
#pragma once
#include "kernels.h"

namespace pamrec {

// The dense layers of the head are small GEMMs (M = B or B*T rows, K and N <= 100).  All three kernels share one
// shape: a CTA of 128 threads owns a 32 x 32 output tile, thread (ty, tx) = (tid / 8, tid % 8) keeps a 2 x 4 patch of
// accumulators, and the two operands sit in shared memory as As[kk][32] / Bs[kk][32] with the contraction index kk
// leading, so one LDS.64 (4 distinct addresses per warp) and one LDS.128 (128 contiguous bytes per warp) feed 8 FMAs.
// Grids are (row tiles) x (groups x column tiles): hundreds of CTAs even at B = 1025, every global load of a tile is
// issued before the first use (the layers are latency-bound, not FLOP-bound).
constexpr int kTM = 32;        // output rows per tile
constexpr int kTN = 32;        // output columns per tile
constexpr int kKMax = 104;     // largest contraction length held in shared memory at once
constexpr int kHT = 128;       // threads per CTA

__device__ __forceinline__ float bn_relu(float z, const float* stat, const float* gamma, const float* beta, int col) {
  float xh = (z - stat[2 * col]) * stat[2 * col + 1];
  return fmaxf(fmaf(gamma[col], xh, beta[col]), 0.f);
}
__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// acc[2][4] += sum_kk As[kk][2ty .. 2ty+1] (x) Bs[kk][4tx .. 4tx+3]
__device__ __forceinline__ void tile_mma(const float* __restrict__ As, const float* __restrict__ Bs, int kk_n, int ty, int tx,
                                         float (&acc)[2][4]) {
#pragma unroll 4
  for (int kk = 0; kk < kk_n; ++kk) {
    const float2 a = *reinterpret_cast<const float2*>(As + kk * kTM + 2 * ty);
    const float4 b = ld4(Bs + kk * kTN + 4 * tx);
    acc[0][0] = fmaf(a.x, b.x, acc[0][0]); acc[0][1] = fmaf(a.x, b.y, acc[0][1]);
    acc[0][2] = fmaf(a.x, b.z, acc[0][2]); acc[0][3] = fmaf(a.x, b.w, acc[0][3]);
    acc[1][0] = fmaf(a.y, b.x, acc[1][0]); acc[1][1] = fmaf(a.y, b.y, acc[1][1]);
    acc[1][2] = fmaf(a.y, b.z, acc[1][2]); acc[1][3] = fmaf(a.y, b.w, acc[1][3]);
  }
}

// Stage rows [m0, m0+32) x columns [c0, c0+cn) of a row-major matrix (leading dimension ld) TRANSPOSED into
// dst[c][32] (c = column offset), zero-filling rows >= rows_valid.  f(value, column offset) is applied on the way.
// Thread i handles row i % 32: the transposed store is bank-conflict free; the strided 16-byte reads hit L1/L2.
template <typename F>
__device__ __forceinline__ void stage_rows_T(float* __restrict__ dst, const float* __restrict__ src, int ld, int rows_valid,
                                             int cn, int tid, F f) {
  const bool vec = ((ld | cn) & 3) == 0 && aligned16(src);
  if (vec) {
    const int n4 = cn >> 2, total = kTM * n4;
    constexpr int IT = (kTM * (kKMax / 4) + kHT - 1) / kHT;
    float4 v[IT];
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      const int i = tid + it * kHT;
      const int r = i % kTM, c4 = i / kTM;
      v[it] = (i < total && r < rows_valid) ? ld4(src + (int64_t)r * ld + 4 * c4) : f4_zero();
    }
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      const int i = tid + it * kHT;
      const int r = i % kTM, c4 = i / kTM;
      if (i < total) {
        const bool ok = r < rows_valid;
        dst[(4 * c4 + 0) * kTM + r] = ok ? f(v[it].x, 4 * c4 + 0) : 0.f;
        dst[(4 * c4 + 1) * kTM + r] = ok ? f(v[it].y, 4 * c4 + 1) : 0.f;
        dst[(4 * c4 + 2) * kTM + r] = ok ? f(v[it].z, 4 * c4 + 2) : 0.f;
        dst[(4 * c4 + 3) * kTM + r] = ok ? f(v[it].w, 4 * c4 + 3) : 0.f;
      }
    }
  } else {
    const int total = kTM * cn;
    for (int i = tid; i < total; i += kHT) {
      const int r = i % kTM, c = i / kTM;
      dst[c * kTM + r] = (r < rows_valid) ? f(src[(int64_t)r * ld + c], c) : 0.f;
    }
  }
}

// dz from (dA, z) with the per-column coefficients of the layer's BN (BnGrad, common.cuh) staged in shared memory:
// co[6c .. 6c+5] = mean, invstd, gamma, beta, S1/n, S2/n  (the two fp64 divisions happen once per column and CTA)
__device__ __forceinline__ void bn_dz_coef(float* __restrict__ co, const BnGrad& g, double count, int col0, int n, int tid) {
  for (int c = tid; c < n; c += kHT) {
    const int cc = col0 + c;
    co[6 * c + 0] = g.stat[2 * cc]; co[6 * c + 1] = g.stat[2 * cc + 1];
    co[6 * c + 2] = g.gamma[cc]; co[6 * c + 3] = g.beta[cc];
    co[6 * c + 4] = (float)(g.bsums[2 * cc] / count); co[6 * c + 5] = (float)(g.bsums[2 * cc + 1] / count);
  }
}
__device__ __forceinline__ float bn_dz(float da, float z, const float* __restrict__ co, int c) {
  const float inv = co[6 * c + 1], ga = co[6 * c + 2];
  const float xh = (z - co[6 * c]) * inv;
  const float dy = fmaf(ga, xh, co[6 * c + 3]) > 0.f ? da : 0.f;
  return ga * inv * (dy - co[6 * c + 4] - xh * co[6 * c + 5]);
}
// stage_rows_T over two matrices with the same layout: dst[c][r] = f(a[r][c], b[r][c], c)
template <typename F>
__device__ __forceinline__ void stage_rows_T2(float* __restrict__ dst, const float* __restrict__ srcA, const float* __restrict__ srcB,
                                              int ld, int rows_valid, int cn, int tid, F f) {
  const bool vec = ((ld | cn) & 3) == 0 && aligned16(srcA) && aligned16(srcB);
  if (vec) {
    const int n4 = cn >> 2, total = kTM * n4;
    constexpr int IT = (kTM * (kKMax / 4) + kHT - 1) / kHT;
#pragma unroll 1
    for (int it0 = 0; it0 < IT; it0 += 4) {             // 4 x 2 float4 in flight per thread
      float4 va[4], vb[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = tid + (it0 + q) * kHT;
        const int r = i % kTM, c4 = i / kTM;
        const bool ok = i < total && r < rows_valid;
        va[q] = ok ? ld4(srcA + (int64_t)r * ld + 4 * c4) : f4_zero();
        vb[q] = ok ? ld4(srcB + (int64_t)r * ld + 4 * c4) : f4_zero();
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = tid + (it0 + q) * kHT;
        const int r = i % kTM, c4 = i / kTM;
        if (i < total) {
          const bool ok = r < rows_valid;
          dst[(4 * c4 + 0) * kTM + r] = ok ? f(va[q].x, vb[q].x, 4 * c4 + 0) : 0.f;
          dst[(4 * c4 + 1) * kTM + r] = ok ? f(va[q].y, vb[q].y, 4 * c4 + 1) : 0.f;
          dst[(4 * c4 + 2) * kTM + r] = ok ? f(va[q].z, vb[q].z, 4 * c4 + 2) : 0.f;
          dst[(4 * c4 + 3) * kTM + r] = ok ? f(va[q].w, vb[q].w, 4 * c4 + 3) : 0.f;
        }
      }
    }
  } else {
    const int total = kTM * cn;
    for (int i = tid; i < total; i += kHT) {
      const int r = i % kTM, c = i / kTM;
      dst[c * kTM + r] = (r < rows_valid) ? f(srcA[(int64_t)r * ld + c], srcB[(int64_t)r * ld + c], c) : 0.f;
    }
  }
}

// shared memory: As | Bs | red (kDenseFwdSmem bytes).  A contraction longer than kKMax (the attention MLP of the sibling models at
// 32 / 8 widths: K = 160) runs in chunks of kKMax: As / Bs hold one chunk and the products accumulate in k order, so a layer with
// K <= kKMax is one chunk with the weight tile staged once per CTA.
constexpr int kDenseFwdSmem = 2 * kKMax * kTM * 4 + 2 * (kHT / 8) * kTN * 8;
__device__ __forceinline__ void dense_fwd_item(const DenseP& p, int M, double* out_sums, int tiles_m, int bx, int gx, int by, unsigned char* smem) {
  float* As = reinterpret_cast<float*>(smem);
  float* Bs = As + kKMax * kTM;
  double (*red)[kHT / 8][kTN] = reinterpret_cast<double (*)[kHT / 8][kTN]>(Bs + kKMax * kTN);
  const int tid = threadIdx.x, ty = tid >> 3, tx = tid & 7;
  const int nchunk = (p.N + kTN - 1) / kTN;
  const int g = by / nchunk, c0 = (by % nchunk) * kTN;
  const int nc = min(kTN, p.N - c0);
  const int xo = p.x_off[g], zo = p.z_off[g] + c0;
  const float* W = p.W + (int64_t)g * p.w_stride;
  const bool one_chunk = p.K <= kKMax;
  // weight tile Bs[k][n] = W[k0+k][c0+n], k < kc
  auto stage_w = [&](int k0, int kc) {
    const bool vec = ((p.N | c0) & 3) == 0 && (nc & 3) == 0 && aligned16(W);
    if (vec) {
      const int n4 = nc >> 2;
      for (int i = tid; i < kc * (kTN / 4); i += kHT) {
        const int k = i / (kTN / 4), q = i % (kTN / 4);
        st4(Bs + k * kTN + 4 * q, q < n4 ? ld4(W + (int64_t)(k0 + k) * p.N + c0 + 4 * q) : f4_zero());
      }
    } else {
      for (int i = tid; i < kc * kTN; i += kHT) {
        const int k = i / kTN, n = i % kTN;
        Bs[i] = n < nc ? W[(int64_t)(k0 + k) * p.N + c0 + n] : 0.f;
      }
    }
  };
  if (one_chunk) stage_w(0, p.K);
  float bias[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) bias[j] = (4 * tx + j < nc) ? p.bias[(int64_t)g * p.b_stride + c0 + 4 * tx + j] : 0.f;
  double cs[4] = {0.0, 0.0, 0.0, 0.0}, cq[4] = {0.0, 0.0, 0.0, 0.0};
  const bool vec_out = ((p.ldz | zo) & 3) == 0 && aligned16(p.Z) && (nc & 3) == 0;
  for (int tm = bx; tm < tiles_m; tm += gx) {
    const int m0 = tm * kTM;
    const int rows = min(kTM, M - m0);
    float acc[2][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < p.K; k0 += kKMax) {
      const int kc = min(kKMax, p.K - k0);
      __syncthreads();                                // previous chunk's / tile's As (and Bs) fully consumed; Bs written (one chunk)
      if (!one_chunk) stage_w(k0, kc);
      const float* X = p.X + (int64_t)m0 * p.ldx + xo + k0;
      if (p.in_stat) {
        const float* st = p.in_stat; const float* ga = p.in_gamma; const float* be = p.in_beta;
        const int xk = xo + k0;
        stage_rows_T(As, X, p.ldx, rows, kc, tid, [=](float v, int k) { return bn_relu(v, st, ga, be, xk + k); });
      } else {
        stage_rows_T(As, X, p.ldx, rows, kc, tid, [](float v, int) { return v; });
      }
      __syncthreads();
      tile_mma(As, Bs, kc, ty, tx, acc);
    }
    // the bias joins the finished product (as tf.matmul + bias does): ONE rounding at the bias's magnitude instead of K of them.
    // It matters where a batch norm follows: a bias of 0.1 in front of a signal of std 5e-4 (the attention MLPs of the sibling
    // models at init) puts every partial sum on a 1.5e-8 grid, and the normalisation then amplifies that by 1 / sqrt(eps) = 100.
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] += bias[j];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int r = 2 * ty + i;
      if (r < rows) {
        float* z = p.Z + (int64_t)(m0 + r) * p.ldz + zo + 4 * tx;
        if (vec_out) { if (4 * tx < nc) st4(z, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3])); }
        else {
#pragma unroll
          for (int j = 0; j < 4; ++j) if (4 * tx + j < nc) z[j] = acc[i][j];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) { cs[j] += (double)acc[i][j]; cq[j] += (double)acc[i][j] * (double)acc[i][j]; }
      }
    }
  }
  if (out_sums) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[0][ty][4 * tx + j] = cs[j]; red[1][ty][4 * tx + j] = cq[j]; }
    __syncthreads();
    if (tid < 2 * kTN) {
      const int which = tid / kTN, n = tid % kTN;
      if (n < nc) {
        double t = 0.0;
#pragma unroll
        for (int y = 0; y < kHT / 8; ++y) t += red[which][y][n];
        atomicAdd(out_sums + 2 * (zo + n) + which, t);
      }
    }
  }
}

// shared memory: As (dZ tile, transposed: As[n][m]) | Bs (Bs[n][kk] = W[k0+kk][n]) | co (BN-backward coefficients of the dZ columns in flight)
constexpr int kDenseDxSmem = 2 * kKMax * kTM * 4 + 6 * kKMax * 4;
__device__ __forceinline__ void dense_dx_item(const DenseDxP& p, int M, double g_count, int bx, int by, unsigned char* smem) {
  float* As = reinterpret_cast<float*>(smem);
  float* Bs = As + kKMax * kTM;
  float* co = Bs + kKMax * kTN;
  const int tid = threadIdx.x, ty = tid >> 3, tx = tid & 7;
  const int kchunk = (p.K + kTN - 1) / kTN;
  const int s = by / kchunk, k0 = (by % kchunk) * kTN;
  const int kc = min(kTN, p.K - k0);
  const int m0 = bx * kTM;
  const int rows = min(kTM, M - m0);
  float acc[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int ci = 0; ci < p.n_contrib[s]; ++ci) {
    const int N = p.Ncon[s][ci], dzo = p.dz_off[s][ci];
    const float* W = p.Wbase + p.w_off[s][ci];
    __syncthreads();
    if (p.g.Z) {
      bn_dz_coef(co, p.g, g_count, dzo, N, tid);
      __syncthreads();
      stage_rows_T2(As, p.dZ + (int64_t)m0 * p.lddz + dzo, p.g.Z + (int64_t)m0 * p.lddz + dzo, p.lddz, rows, N, tid,
                    [&](float da, float z, int c) { return bn_dz(da, z, co, c); });
    } else {
      stage_rows_T(As, p.dZ + (int64_t)m0 * p.lddz + dzo, p.lddz, rows, N, tid, [](float v, int) { return v; });
    }
    // rows of W are the "rows" to transpose: Bs[n][kk] = W[(k0+kk)*N + n]
    stage_rows_T(Bs, W + (int64_t)k0 * N, N, kc, N, tid, [](float v, int) { return v; });
    __syncthreads();
    tile_mma(As, Bs, N, ty, tx, acc);
  }
  const int oo = p.out_off[s] + k0;
  const bool vec_out = ((p.lddx | oo) & 3) == 0 && aligned16(p.dX) && (kc & 3) == 0;
  double s1[4] = {0.0, 0.0, 0.0, 0.0}, s2[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int r = 2 * ty + i;
    if (r < rows) {
      float* o = p.dX + (int64_t)(m0 + r) * p.lddx + oo + 4 * tx;
      if (p.accumulate) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (4 * tx + j < kc) acc[i][j] += o[j];
      }
      if (vec_out) { if (4 * tx < kc) st4(o, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3])); }
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (4 * tx + j < kc) o[j] = acc[i][j];
      }
      if (p.o.Z) {                                     // BN-backward sums of the buffer just produced
        const float* z = p.o.Z + (int64_t)(m0 + r) * p.lddx + oo + 4 * tx;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (4 * tx + j < kc) {
            const int c = oo + 4 * tx + j;
            const float xh = (z[j] - p.o.stat[2 * c]) * p.o.stat[2 * c + 1];
            const float dy = fmaf(p.o.gamma[c], xh, p.o.beta[c]) > 0.f ? acc[i][j] : 0.f;
            s1[j] += (double)dy;
            s2[j] += (double)dy * (double)xh;
          }
      }
    }
  }
  if (p.o.Z) {
    double* red = reinterpret_cast<double*>(As);       // [2][16][32] doubles = 8 KB, As is free now
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[ty * kTN + 4 * tx + j] = s1[j]; red[(kHT / 8) * kTN + ty * kTN + 4 * tx + j] = s2[j]; }
    __syncthreads();
    if (tid < 2 * kTN) {
      const int which = tid / kTN, n = tid % kTN;
      if (n < kc) {
        double tsum = 0.0;
#pragma unroll
        for (int y = 0; y < kHT / 8; ++y) tsum += red[which * (kHT / 8) * kTN + y * kTN + n];
        atomicAdd(p.o.bsums + 2 * (oo + n) + which, tsum);
      }
    }
  }
}

// shared memory: As[r][kk] = act(X[m0+r, xo+k0+kk]) | Bs[r][nn] = dZ[m0+r, zo+n0+nn] | co (BN-backward coefficients of this tile's dZ columns)
constexpr int kDenseDwSmem = 2 * kTM * kTM * 4 + 6 * kTN * 4;
__device__ __forceinline__ void dense_dw_item(const DenseDwP& p, int M, double g_count, int rows_per_cta, int bx, int by, unsigned char* smem) {
  float* As = reinterpret_cast<float*>(smem);
  float* Bs = As + kTM * kTM;
  float* co = Bs + kTM * kTN;
  const int tid = threadIdx.x, ty = tid >> 3, tx = tid & 7;
  const int ktiles = (p.K + kTM - 1) / kTM, ntiles = (p.N + kTN - 1) / kTN;
  int y = by;
  const int nt = y % ntiles; y /= ntiles;
  const int kt = y % ktiles;
  const int g = y / ktiles;
  const int k0 = kt * kTM, n0 = nt * kTN;
  const int kc = min(kTM, p.K - k0), nc = min(kTN, p.N - n0);
  const int xo = p.x_off[g] + k0, zo = p.z_off[g] + n0;
  const int m_begin = bx * rows_per_cta, m_end = min(M, m_begin + rows_per_cta);
  const bool vecA = ((p.ldx | xo) & 3) == 0 && (kc & 3) == 0 && aligned16(p.X);
  const bool vecB = ((p.lddz | zo) & 3) == 0 && (nc & 3) == 0 && aligned16(p.dZ);
  float acc[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float dbv = 0.f;
  if (p.g.Z) bn_dz_coef(co, p.g, g_count, zo, nc, tid);       // visible after the first barrier of the loop
  for (int m0 = m_begin; m0 < m_end; m0 += kTM) {
    const int rows = min(kTM, m_end - m0);
    __syncthreads();
    // each thread stages 2 float4 (or 8 scalars) of each operand: row r = i / 8, quad q = i % 8
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int i = tid + it * kHT;
      const int r = i >> 3, q = i & 7;
      float4 a = f4_zero(), b = f4_zero();
      if (r < rows) {
        const float* xa = p.X + (int64_t)(m0 + r) * p.ldx + xo + 4 * q;
        const float* zb = p.dZ + (int64_t)(m0 + r) * p.lddz + zo + 4 * q;
        if (vecA) { if (4 * q < kc) a = ld4(xa); }
        else {
          if (4 * q + 0 < kc) a.x = xa[0];
          if (4 * q + 1 < kc) a.y = xa[1];
          if (4 * q + 2 < kc) a.z = xa[2];
          if (4 * q + 3 < kc) a.w = xa[3];
        }
        if (p.in_stat) {
          const int col = xo + 4 * q;
          if (4 * q + 0 < kc) a.x = bn_relu(a.x, p.in_stat, p.in_gamma, p.in_beta, col + 0);
          if (4 * q + 1 < kc) a.y = bn_relu(a.y, p.in_stat, p.in_gamma, p.in_beta, col + 1);
          if (4 * q + 2 < kc) a.z = bn_relu(a.z, p.in_stat, p.in_gamma, p.in_beta, col + 2);
          if (4 * q + 3 < kc) a.w = bn_relu(a.w, p.in_stat, p.in_gamma, p.in_beta, col + 3);
        }
        if (vecB) { if (4 * q < nc) b = ld4(zb); }
        else {
          if (4 * q + 0 < nc) b.x = zb[0];
          if (4 * q + 1 < nc) b.y = zb[1];
          if (4 * q + 2 < nc) b.z = zb[2];
          if (4 * q + 3 < nc) b.w = zb[3];
        }
        if (p.g.Z) {
          const float* zz = p.g.Z + (int64_t)(m0 + r) * p.lddz + zo + 4 * q;
          if (4 * q + 0 < nc) b.x = bn_dz(b.x, zz[0], co, 4 * q + 0);
          if (4 * q + 1 < nc) b.y = bn_dz(b.y, zz[1], co, 4 * q + 1);
          if (4 * q + 2 < nc) b.z = bn_dz(b.z, zz[2], co, 4 * q + 2);
          if (4 * q + 3 < nc) b.w = bn_dz(b.w, zz[3], co, 4 * q + 3);
        }
      }
      st4(As + r * kTM + 4 * q, a);
      st4(Bs + r * kTN + 4 * q, b);
    }
    __syncthreads();
    tile_mma(As, Bs, kTM, ty, tx, acc);       // rows beyond `rows` are zero-filled
    if (kt == 0 && tid < kTN) {
#pragma unroll 8
      for (int r = 0; r < kTM; ++r) dbv += Bs[r * kTN + tid];
    }
  }
  float* dW = p.dW + (int64_t)g * p.w_stride;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int k = 2 * ty + i;
    if (k < kc) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * tx + j < nc) atomicAdd(dW + (int64_t)(k0 + k) * p.N + n0 + 4 * tx + j, acc[i][j]);
    }
  }
  if (kt == 0 && tid < nc) atomicAdd(p.db + (int64_t)g * p.b_stride + n0 + tid, dbv);
  if (p.g_dgamma && bx == 0 && by == 0) {
    for (int c = tid; c < p.g_C; c += kHT) {
      p.g_dbeta[c] += (float)p.g.bsums[2 * c] * p.g_scale;
      p.g_dgamma[c] += (float)p.g.bsums[2 * c + 1] * p.g_scale;
    }
  }
}


// grid decompositions shared by the stand-alone launchers and the persistent kernels: `cap_ctas` ~ CTAs that fill the GPU
struct FwdGrid { int tiles_m, ny, gx; };
__host__ __device__ inline FwdGrid dense_fwd_grid(int M, int n_groups, int N, int cap_ctas) {
  FwdGrid g;
  g.tiles_m = (M + kTM - 1) / kTM;
  g.ny = n_groups * ((N + kTN - 1) / kTN);
  const int cap = (cap_ctas + g.ny - 1) / g.ny;          // enough CTAs to fill the GPU; long matrices loop over row tiles
  const int per_cta = (g.tiles_m + cap - 1) / cap;
  g.gx = per_cta > 0 ? (g.tiles_m + per_cta - 1) / per_cta : 0;
  return g;
}
struct DxGrid { int gx, ny; };
__host__ __device__ inline DxGrid dense_dx_grid(int M, int n_slices, int K) {
  DxGrid g;
  g.gx = (M + kTM - 1) / kTM;
  g.ny = n_slices * ((K + kTN - 1) / kTN);
  return g;
}
struct DwGrid { int chunks, ny, rows_per_cta; };
__host__ __device__ inline DwGrid dense_dw_grid(int M, int n_groups, int K, int N, int cap_ctas) {
  DwGrid g;
  g.ny = n_groups * ((K + kTM - 1) / kTM) * ((N + kTN - 1) / kTN);
  int chunks = (cap_ctas + g.ny - 1) / g.ny;                    // row chunks so that the grid fills the GPU
  const int max_chunks = (M + kTM - 1) / kTM;
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  g.rows_per_cta = ((M + chunks - 1) / chunks + kTM - 1) / kTM * kTM;
  g.chunks = g.rows_per_cta > 0 ? (M + g.rows_per_cta - 1) / g.rows_per_cta : 0;
  return g;
}

}  // namespace pamrec
