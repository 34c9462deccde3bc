// Attention maps of the encoder blocks (pamrec_attention, api_attn.inl): the softmax probabilities of every (query, key) pair of a
// sample, recomputed after the scoring forward pass from what it saved - the queries and keys of each block and the row statistics
// (m, l) of its softmax:
//
//   P[q, k] = exp(s_qk - m_q) / l_q   on a live key,   0 on a masked key,   1 / l_q (= 1 / T) in a sample without live keys.
//
// The scores s_qk = q . k / sqrt(S) run on the tensor cores as the error-compensated 3xTF32 product of kernels_attn_mma.cu, with
// its operand split and accumulation order (mma_rows_t).  Where PAMRec's forward ran that kernel (T <= 128) the scores are the
// forward's own bit for bit, so the largest weight of a row is exactly 1 / l_q.  Where the forward summed in FP32 FMAs (PAMRec above
// T = 128, SASRec) a score differs from the forward's by fp32 rounding only (~1e-7 relative).
//
// Why tensor cores: at long_b4095_t200 the maps are 1.31 GB (0.17 ms at 7.7 TB/s) but the scores are 26 GFLOP, which alone take
// 0.34 ms at the FP32 FMA peak.  Measured on a B200 (DESIGN.md): 0.94 ms there, neither at the store floor nor at an FMA or MMA
// rate limit.
//
// One CTA per (64 query rows, sample, block), four warps of 16 query rows.  The sample's keys sit in shared memory (zero padded to
// a multiple of 8 rows and of 8 columns); small CTAs let several (sample, block) pairs share an SM, so one CTA's key staging overlaps
// the others' products and stores.  Per 8-key tile a warp forms the 16 x 8 score fragment, turns it into probabilities in
// registers and stores it: rows g and g + 8 of the tile, 8 consecutive floats each, so a tile's row segment is one 32-byte sector and
// a warp writes its 16 rows front to back.
#include "kernels.h"
#include "mma.cuh"

namespace pamrec {

// shared-memory row stride of the keys: >= the padded width, and 4 x odd so that the fragment loads (bank 4 odd g + t) never conflict
template <int S> constexpr int map_stride() { return S == 40 ? 44 : 28; }

// c[4] += A[16 x 8 KS] . R^T for the 8 key rows n0 .. n0 + 7 of R: the three split terms as three chains, small terms added last
// (kernels_attn_mma.cu:mma_rows_t, the same operations in the same order)
template <int KS, int ST>
__device__ __forceinline__ void map_rows_t(float (&c)[4], const uint32_t (&ahi)[KS][4], const uint32_t (&alo)[KS][4],
                                           const float* __restrict__ R, int n0, int g, int t) {
  const float* r = R + (n0 + g) * ST + t;
  float d1[4] = {0.f, 0.f, 0.f, 0.f}, d2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k0 = 0; k0 < KS; ++k0) {
    uint32_t bh[2], bl[2];
    split_tf32(r[8 * k0], bh[0], bl[0]);
    split_tf32(r[8 * k0 + 4], bh[1], bl[1]);
    mma_tf32(d1, alo[k0], bh);
    mma_tf32(d2, ahi[k0], bl);
    mma_tf32(c, ahi[k0], bh);
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) c[e] += d1[e] + d2[e];
}

// grid: (samples x query-row groups of kMapRows, blocks); blockIdx.y + blk0 = the encoder block.  With a.maps null only the CTA and
// warp holding block 1's read-out row (SASRec's pool) compute.
constexpr int kMapWarps = 4, kMapRows = 16 * kMapWarps;
template <int S, bool SAS>
__global__ void __launch_bounds__(32 * kMapWarps) k_attn_map(const AttnMapArgs a, int blk0) {
  constexpr int KS = (S + 7) / 8, ST = map_stride<S>();
  extern __shared__ __align__(16) float sm[];
  __shared__ int s_nl;
  const int T = a.T, Tp = (T + 7) & ~7, ng = (T + kMapRows - 1) / kMapRows, b = blockIdx.x / ng, grp = blockIdx.x % ng;
  const int blk = blk0 + blockIdx.y, tid = threadIdx.x;
  float* Ks = sm;                                         // [Tp][ST] keys
  float* Ms = Ks + Tp * ST;                               // [T][2] m, 1 / l
  int* live = reinterpret_cast<int*>(Ms + 2 * T);         // [Tp]
  const int64_t base = (int64_t)b * T;
  const float* __restrict__ ML = blk ? a.ML[1] : a.ML[0];
  const float* __restrict__ Q = blk ? a.Q[1] : a.Q[0];
  const float* __restrict__ K = blk ? a.K[1] : a.K[0];
  if (tid == 0) s_nl = 0;
  __syncthreads();
  int cnt = 0;
  for (int j = tid; j < Tp; j += 32 * kMapWarps) {
    int lv = 0;
    if (j < T) {
      const int mk = a.mask[base + j];
      lv = SAS ? (mk == 1) : (mk != 0);
      Ms[2 * j] = ML[2 * (base + j)];
      Ms[2 * j + 1] = 1.0f / ML[2 * (base + j) + 1];
    }
    live[j] = lv;
    cnt += lv;
  }
  if (cnt) atomicAdd(&s_nl, cnt);
  __syncthreads();
  const int nl = s_nl;
  const int rsel = nl > 0 ? nl - 1 : 0;                   // the row k_sas_final_fwd reads (length - 1; row 0 of an all-uniform map)
  if (!a.maps && grp != rsel / kMapRows) return;
  // the CTAs of one (sample, block) are adjacent in the grid: the key rows come from L2 after the first
  for (int i = tid; i < Tp * (ST / 4); i += 32 * kMapWarps) {
    const int r = i / (ST / 4), c = i % (ST / 4);
    st4(Ks + r * ST + 4 * c, (r < T && 4 * c < S) ? ld4(K + (base + r) * a.ld + 4 * c) : f4_zero());
  }
  __syncthreads();
  const int w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int r0 = kMapRows * grp + 16 * w;
  if (r0 >= T || (!a.maps && r0 != rsel / 16 * 16)) return;
  const int ra = r0 + g, rb = ra + 8;
  uint32_t qhi[KS][4], qlo[KS][4];
#pragma unroll
  for (int k0 = 0; k0 < KS; ++k0) {
    const int c = 8 * k0 + t;
    auto q = [&](int r, int col) { return (r < T && col < S) ? Q[(base + r) * a.ld + col] : 0.f; };
    split_tf32(q(ra, c), qhi[k0][0], qlo[k0][0]);
    split_tf32(q(rb, c), qhi[k0][1], qlo[k0][1]);
    split_tf32(q(ra, c + 4), qhi[k0][2], qlo[k0][2]);
    split_tf32(q(rb, c + 4), qhi[k0][3], qlo[k0][3]);
  }
  const float ma = ra < T ? Ms[2 * ra] : 0.f, ia = ra < T ? Ms[2 * ra + 1] : 0.f;
  const float mb = rb < T ? Ms[2 * rb] : 0.f, ib = rb < T ? Ms[2 * rb + 1] : 0.f;
  const float scale = SAS ? (S == 40 ? 0.15811388300841897f : 0.22360679774997896f)     // kernels_sasrec.cu:sas_scale
                          : 1.0f / sqrtf((float)S);                                      // kernels_attn_mma.cu:rscale
  float* rowa = a.maps ? a.maps + (((int64_t)b * 2 + blk) * T + ra) * T : nullptr;
  float* rowb = rowa ? rowa + 8 * (int64_t)T : nullptr;
  float* pool = (SAS && blk == 1) ? a.pool + base : nullptr;
  const bool even = (T & 1) == 0;
  for (int n0 = 0; n0 < Tp; n0 += 8) {
    float c[4] = {0.f, 0.f, 0.f, 0.f};
    map_rows_t<KS, ST>(c, qhi, qlo, Ks, n0, g, t);
    const int k = n0 + 2 * t;
    float p[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float m = e < 2 ? ma : mb, il = e < 2 ? ia : ib;
      p[e] = nl == 0 ? il : (live[k + (e & 1)] ? expf(c[e] * scale - m) * il : 0.f);
    }
    if (rowa) {
      if (even && k < T) {                                 // T even: k + 1 < T too, and the pair is 8-byte aligned
        if (ra < T) *reinterpret_cast<float2*>(rowa + k) = make_float2(p[0], p[1]);
        if (rb < T) *reinterpret_cast<float2*>(rowb + k) = make_float2(p[2], p[3]);
      } else {
        if (ra < T && k < T) rowa[k] = p[0];
        if (ra < T && k + 1 < T) rowa[k + 1] = p[1];
        if (rb < T && k < T) rowb[k] = p[2];
        if (rb < T && k + 1 < T) rowb[k + 1] = p[3];
      }
    }
    if (pool) {
      if (ra == rsel) { if (k < T) pool[k] = p[0]; if (k + 1 < T) pool[k + 1] = p[1]; }
      if (rb == rsel) { if (k < T) pool[k] = p[2]; if (k + 1 < T) pool[k + 1] = p[3]; }
    }
  }
}

void launch_attn_maps(const AttnMapArgs& a, int S, bool sasrec, cudaStream_t st) {
  PAMREC_PROF("attn_maps", 1, st);
  if (a.B == 0 || (!a.maps && !(sasrec && a.pool))) return;
  const int nblk = a.maps ? 2 : 1, Tp = (a.T + 7) & ~7;
  const dim3 grid((unsigned)(a.B * ((a.T + kMapRows - 1) / kMapRows)), nblk);
  const size_t smem = ((size_t)Tp * map_stride<40>() + 3 * (size_t)Tp) * sizeof(float);   // 47 KB at T = 256: below 48 KB
  const int threads = 32 * kMapWarps;
  if (!sasrec) k_attn_map<kD, false><<<grid, threads, smem, st>>>(a, 2 - nblk);
  else if (S == 40) k_attn_map<40, true><<<grid, threads, smem, st>>>(a, 2 - nblk);
  else k_attn_map<20, true><<<grid, threads, smem, st>>>(a, 2 - nblk);
}

}  // namespace pamrec
