// Gradient all-reduce over NVLink peer memory (k_xr_*), through the exchange region of the mailboxes that every rank maps from its
// peers (cudaIpc, api.cu).
#include "kernels.h"

namespace pamrec {

__device__ __forceinline__ void st_flag(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_flag(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ------------------------------------------------------------------------------------------ gradient all-reduce over peer memory
// Region layout (kernels.h): [0, 256) flags A (contribution of rank p is complete), [256, 512) flags B (rank p has written its
// slice of the result everywhere), scalars [rank][kXrScalars] doubles, contribution `xbuf` [cap], result `rbuf` [cap].
// k_xr_pack: dense gradients -> front of the own contribution (the replicated tables' gradient tables are produced there
// directly), own scalars -> every peer; the last CTA publishes flag A.  k_xr_reduce: wait for every flag A, sum the own slice
// over the ranks in rank order (16-byte loads over NVLink), store the sums into every rank's result buffer; the last CTA
// publishes flag B.  k_xr_finish: wait for every flag B, copy the dense part of the result back, sum the scalars.
// Every rank computes each element exactly once and all ranks receive the same bits.
namespace {
constexpr int kXrThreads = 256;
__device__ __forceinline__ uint32_t* xr_flags(char* region, int which) { return reinterpret_cast<uint32_t*>(region + 256 * which); }
__device__ __forceinline__ double* xr_scal(char* region) { return reinterpret_cast<double*>(region + 512); }
__device__ __forceinline__ float* xr_x(char* region) { return reinterpret_cast<float*>(region + 512 + kP2PMaxWorld * kXrScalars * sizeof(double)); }
__device__ __forceinline__ float4 ld_sys4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_sys4(float* p, const float4& v) {
  asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// all CTAs of the grid have made their writes visible system-wide: the last one to arrive returns true (and resets the counter)
__device__ __forceinline__ bool xr_last_cta(unsigned* counter) {
  __shared__ bool last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicInc(counter, gridDim.x - 1) == gridDim.x - 1;
  __syncthreads();
  return last;
}
__device__ __forceinline__ void xr_wait(const XrArgs& a, int which) {
  if (threadIdx.x < a.world) {
    const uint32_t* f = xr_flags(a.peer[a.rank], which) + threadIdx.x;
    uint32_t spins = 0;
    while ((int32_t)(ld_flag(f) - a.epoch) < 0) {
      if (++spins > (1u << 24)) { *a.err = 200u + (uint32_t)which; break; }
      __nanosleep(40);
    }
  }
  __syncthreads();
}
__global__ void __launch_bounds__(kXrThreads) k_xr_pack(const XrArgs a) {
  float* x = xr_x(a.peer[a.rank]);
  for (int64_t i = (int64_t)blockIdx.x * kXrThreads + threadIdx.x; i < a.n_dense; i += (int64_t)gridDim.x * kXrThreads) x[i] = a.dense_grad[i];
  if (blockIdx.x == 0) {
    const int n0 = a.n_scalars[0], n = n0 + a.n_scalars[1];
    for (int i = threadIdx.x; i < n * a.world; i += kXrThreads) {
      const int p = i / n, k = i % n;
      xr_scal(a.peer[p])[a.rank * kXrScalars + k] = k < n0 ? a.scalars[0][k] : a.scalars[1][k - n0];
    }
  }
  if (xr_last_cta(a.counter) && threadIdx.x < a.world) st_flag(xr_flags(a.peer[threadIdx.x], 0) + a.rank, a.epoch);
}
__global__ void __launch_bounds__(kXrThreads) k_xr_reduce(const XrArgs a) {
  xr_wait(a, 0);
  const int64_t slice = a.cap / a.world, q0 = (int64_t)a.rank * slice / 4, q1 = q0 + slice / 4;
  for (int64_t q = q0 + (int64_t)blockIdx.x * kXrThreads + threadIdx.x; q < q1; q += (int64_t)gridDim.x * kXrThreads) {
    float4 v[kP2PMaxWorld];
#pragma unroll
    for (int p = 0; p < kP2PMaxWorld; ++p) if (p < a.world) v[p] = ld_sys4(xr_x(a.peer[p]) + 4 * q);
    float4 s = v[0];
#pragma unroll
    for (int p = 1; p < kP2PMaxWorld; ++p) if (p < a.world) { s.x += v[p].x; s.y += v[p].y; s.z += v[p].z; s.w += v[p].w; }
#pragma unroll
    for (int p = 0; p < kP2PMaxWorld; ++p) if (p < a.world) st_sys4(xr_x(a.peer[p]) + a.cap + 4 * q, s);
  }
  if (xr_last_cta(a.counter + 1) && threadIdx.x < a.world) st_flag(xr_flags(a.peer[threadIdx.x], 1) + a.rank, a.epoch);
}
__global__ void __launch_bounds__(kXrThreads) k_xr_finish(const XrArgs a, float* __restrict__ dense_out) {
  xr_wait(a, 1);
  const float* r = xr_x(a.peer[a.rank]) + a.cap;
  for (int64_t i = (int64_t)blockIdx.x * kXrThreads + threadIdx.x; i < a.n_dense; i += (int64_t)gridDim.x * kXrThreads) dense_out[i] = __ldcg(r + i);
  if (blockIdx.x == 0) {
    const int n0 = a.n_scalars[0], n = n0 + a.n_scalars[1];
    if ((int)threadIdx.x < n) {
      const int k = threadIdx.x;
      double s = 0.0;
      for (int p = 0; p < a.world; ++p) s += __ldcg(xr_scal(a.peer[a.rank]) + p * kXrScalars + k);
      if (k < n0) a.scalars[0][k] = s; else a.scalars[1][k - n0] = s;
    }
  }
}
}  // namespace

void launch_xr_allreduce(const XrArgs& a, float* dense_grad_out, cudaStream_t st) {
  PAMREC_PROF("allreduce_grads", 3, st);
  const int g_pack = 32;
  const int64_t quads = a.cap / a.world / 4;
  int g_red = (int)((quads + kXrThreads - 1) / kXrThreads);
  g_red = g_red < 1 ? 1 : (g_red > 64 ? 64 : g_red);
  k_xr_pack<<<g_pack, kXrThreads, 0, st>>>(a);
  k_xr_reduce<<<g_red, kXrThreads, 0, st>>>(a);
  k_xr_finish<<<g_pack, kXrThreads, 0, st>>>(a, dense_grad_out);
}

}  // namespace pamrec
