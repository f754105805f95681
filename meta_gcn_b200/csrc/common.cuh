// Shared helpers for the sm_100a kernels of libmgcn.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "mgcn.h"

namespace mgcn {

extern std::atomic<long long> g_launch_count;

// SM count of the CURRENT device (B200: 148 = 2 dies x 74), queried once per device and cached; grids of the
// persistent kernels are sized from it.  Falls back to 148 if the query fails.
inline int num_sms() {
  static std::atomic<int> cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int v = cache[dev].load(std::memory_order_relaxed);
  if (v > 0) return v;
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
  cache[dev].store(v, std::memory_order_relaxed);
  return v;
}
#define kNumSMs (::mgcn::num_sms())

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// carve a sub-buffer out of a workspace; with base == nullptr only the running size is advanced
struct WorkspaceCarver {
  char* base;
  size_t off = 0;
  explicit WorkspaceCarver(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
  size_t bytes() const { return align_up(off, 256); }
};

// ---- L2 residency hints -------------------------------------------------------------------------
// Measured (profiles/r1_layer_summary.md): with plain loads the aggregation kernels read 1.5x their
// compulsory DRAM bytes — the index / descriptor / tile streams and the output stores push the
// gathered feature rows (the only data with reuse) out of L2.  Streams are therefore tagged
// evict-first and bypass L1; gathered rows keep the default policy.
#ifdef __CUDACC__
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ld_f4_hint(const float* p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ int4 ld_i4_hint(const int4* p, uint64_t pol) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ int ld_i32_hint(const int32_t* p, uint64_t pol) {
  int r;
  // allocates in L1: the batches of one row share sectors
  asm volatile("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void st_f4_hint(float* p, float4 v, uint64_t pol) {
  asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async16_hint(void* smem_dst, const void* gsrc, int src_bytes, uint64_t pol) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2, %3;\n"
               :: "r"(d), "l"(gsrc), "r"(src_bytes), "l"(pol) : "memory");
}
#endif

// H = 32 plain aggregation on the flat work-ordered gather (gcn_layer.cu)
int launch_agg_flat32(const mgcn_csr_t* g, const float* x, const float* post, int act, float* out,
                      float* partial, bool hubs, void* stream);

// tcgen05 row-local backward of the hidden-32 layer (gcn_layer_tc.cu)
size_t bwd_tc_workspace_floats(int64_t N);
int launch_layer_bwd_tc(const float* dxw, const float* gy, const float* x, const float* x_scale, const float* w, const float* res_w,
                        const uint32_t* hmask_prev, const float* post, int64_t N, float* gy_prev, float* gs_prev,
                        float* dw, float* d_res_w, float* d_res_b, float* ws, void* stream,
                        const uint32_t* hmask_cur = nullptr, float bias_scale = 1.f, float* d_bias = nullptr);
// floats the launch above needs beyond bwd_tc_workspace_floats when d_bias is given (the masked column sum's partials)
size_t bwd_tc_bias_workspace_floats(int64_t N);
// dW / dR from per-CTA partials [P][128][32] of the transposed tcgen05 products, fixed order (gcn_layer_tc.cu)
int launch_bwd_tc_reduce(const float* part, int P, float* dw, float* d_res_w, const float* part_b, int Pb,
                         float* d_res_b, void* stream);
// d_bias[c] = scale * sum_i bit c of bits[i] * gy[i][c] over [N][32], two fixed-order levels (gcn_layer_tc.cu)
size_t mask_bits_colsum_workspace_floats(int64_t N);
int launch_mask_bits_colsum(const float* gy, const uint32_t* bits, float scale, int64_t N, float* d_bias, float* ws,
                            void* stream);
// narrow-side dense transforms (dense_narrow.cu)
bool narrow_linear_applies(int64_t Hi, int64_t Ho, const float* x, const float* xmask, const float* add,
                           const float* y);
int launch_narrow_linear(const float* x, const float* xmask, int64_t N, int64_t Hi, const float* w,
                         int64_t w_sk, int64_t w_sc, int64_t Ho, const float* bias, const float* add,
                         int act, const float* row_scale, float* y, void* stream);
bool narrow_wgrad_applies(int64_t Hi, int64_t Ho, const float* x, const float* g, const float* gmask);
size_t narrow_wgrad_blocks(int64_t N);
int launch_narrow_wgrad(const float* x, int64_t N, int64_t Hi, const float* g, const float* gmask,
                        int64_t Ho, float* dw, int64_t dw_sk, int64_t dw_sc, float* db, float* part,
                        float* part_db, void* stream);
// wide weight gradient on tcgen05 (wgrad_wide.cu)
bool wide_wgrad_applies(int64_t N, int64_t Hi, int64_t Ho, const float* x, const float* g, const float* gmask);
int wide_wgrad_splits(int64_t Hi);
int launch_wide_wgrad(const float* x, int64_t N, int64_t Hi, const float* g, const float* gmask, int64_t Ho,
                      float* dw, int64_t dw_sk, int64_t dw_sc, float* db, float* partial, float* partial_b,
                      void* stream);
// out[k*sk + c*sc] = sum_p partial[p*count + k*Hc + c], fixed order
int launch_reduce_partials(const float* partial, int P, int count, int Hc, float* out, int64_t sk,
                           int64_t sc, void* stream);

}  // namespace mgcn

// Launch + count + error check.  Used inside functions returning int.
#define MGCN_LAUNCH(kernel, grid, block, smem, stream, ...)                          \
  do {                                                                               \
    kernel<<<(grid), (block), (smem), static_cast<cudaStream_t>(stream)>>>(__VA_ARGS__); \
    ::mgcn::g_launch_count.fetch_add(1, std::memory_order_relaxed);                  \
    cudaError_t mgcn_err__ = cudaGetLastError();                                     \
    if (mgcn_err__ != cudaSuccess) return static_cast<int>(mgcn_err__);              \
  } while (0)

#define MGCN_CHECK_CUDA(expr)                                       \
  do {                                                              \
    cudaError_t mgcn_err__ = (expr);                                \
    if (mgcn_err__ != cudaSuccess) return static_cast<int>(mgcn_err__); \
  } while (0)

#define MGCN_REQUIRE(cond, code) \
  do {                           \
    if (!(cond)) return (code);  \
  } while (0)
