// Dropout of the residual GCN stack (gcn_model.py:92: xo = dropout(relu(agg)) before the residual add).
//
//   k_dropout_keep_bits  keep[l][n][w] bit b = column 32 w + b of row n in layer l is kept.  One thread per word:
//                        4 Philox4x32-10 calls (csrc/philox.cuh), each output word split into two 16-bit draws.
//                        The word depends on (seed, l, n, w) only — the forward kernels that read it fill their
//                        tiles in completion order, so the mask must not depend on which thread asks for it.
//   k_dropout_apply      h[n,c] = keep bit ? h[n,c] * scale : 0, in place (the generic stack, widths 16..128).
// The hidden-32 stack applies the bits in the epilogues of its forward kernels instead (gcn_fwd_tc.cu, gcn_layer.cu),
// where the cleared bits also clear the ReLU mask word the backward reads.
#include <cmath>

#include "common.cuh"
#include "philox.cuh"

namespace mgcn {

__global__ void __launch_bounds__(256) k_dropout_keep_bits(const int64_t* __restrict__ seed, uint32_t per_layer,
                                                           uint32_t W, uint32_t t, uint32_t* __restrict__ keep) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;   // per_layer = N W < 2^31
  if (i >= per_layer) return;
  const uint32_t l = blockIdx.y;
  const uint32_t n = i / W, w = i - n * W;
  const uint64_t s = (uint64_t)__ldg(seed);
  const uint32_t k0 = (uint32_t)s, k1 = (uint32_t)(s >> 32);
  uint32_t bits = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint4 r = philox4x32_10(make_uint4(n, l, 4 * w + j, 0u), k0, k1);
    const uint32_t v[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      bits |= ((v[q] & 0xffffu) >= t ? 1u : 0u) << (8 * j + 2 * q);
      bits |= ((v[q] >> 16) >= t ? 1u : 0u) << (8 * j + 2 * q + 1);
    }
  }
  keep[(int64_t)l * per_layer + i] = bits;
}

__global__ void __launch_bounds__(256) k_dropout_apply(float* __restrict__ h, const uint32_t* __restrict__ keep,
                                                       int64_t N, int H, int W, float scale) {
  const int64_t total = N * (H / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / (H / 4);
    const int c = (int)(i - row * (H / 4)) * 4;
    const uint32_t b = __ldg(keep + row * W + (c >> 5)) >> (c & 31);
    float4 v = reinterpret_cast<float4*>(h)[i];
    v.x = (b & 1u) ? __fmul_rn(v.x, scale) : 0.f;
    v.y = (b & 2u) ? __fmul_rn(v.y, scale) : 0.f;
    v.z = (b & 4u) ? __fmul_rn(v.z, scale) : 0.f;
    v.w = (b & 8u) ? __fmul_rn(v.w, scale) : 0.f;
    reinterpret_cast<float4*>(h)[i] = v;
  }
}

}  // namespace mgcn

using namespace mgcn;

extern "C" int mgcn_dropout_keep_bits(const int64_t* seed, int64_t L, int64_t N, int64_t W, float p, uint32_t* keep,
                                      void* stream) {
  MGCN_REQUIRE(L >= 0 && L <= 65535 && N >= 0 && W >= 1 && W <= 1024, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N * W < (int64_t(1) << 31), MGCN_ERR_RANGE);
  MGCN_REQUIRE(p >= 0.f && p <= 1.f, MGCN_ERR_SHAPE);   // also refuses NaN
  const int64_t t = std::llrint((double)p * 65536.0);
  MGCN_REQUIRE(t < 65536, MGCN_ERR_SHAPE);              // nothing kept: no scale 1 / (1 - p) exists
  if (L == 0 || N == 0) return MGCN_OK;
  MGCN_REQUIRE(seed && keep, MGCN_ERR_NULL);
  const dim3 grid((unsigned)ceil_div(N * W, 256), (unsigned)L);
  MGCN_LAUNCH(k_dropout_keep_bits, grid, 256, 0, stream, seed, (uint32_t)(N * W), (uint32_t)W, (uint32_t)t, keep);
  return MGCN_OK;
}

extern "C" int mgcn_dropout_apply(float* h, const uint32_t* keep, int64_t N, int64_t H, int64_t W, float scale,
                                  void* stream) {
  MGCN_REQUIRE(H > 0 && H % 4 == 0 && W >= (H + 31) / 32 && W <= 1024, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N >= 0 && N < (int64_t(1) << 31), MGCN_ERR_RANGE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(h && keep, MGCN_ERR_NULL);
  MGCN_REQUIRE(aligned16(h), MGCN_ERR_ALIGN);
  int64_t blocks = ceil_div(N * (H / 4), 256);
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  MGCN_LAUNCH(k_dropout_apply, (unsigned)blocks, 256, 0, stream, h, keep, N, (int)H, (int)W, scale);
  return MGCN_OK;
}
