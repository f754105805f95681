// Cross-entropy over node logits — nn.CrossEntropyLoss()(x, batch.y.long()) of
// train_botnet.py:225,287 — as two small deterministic kernels (fixed-order two-stage sum), so
// the step has no single-block torch reduction over 3.6 M rows on its critical path.
#include <limits>

#include "common.cuh"

namespace mgcn {

constexpr int kCeThreads = 256;

// log1p(t) - (z_y - m) with t = sum over the classes other than the (first) argmax of exp(z_c - m): the term
// exp(z_argmax - m) = 1 is left out, so the small NLL of a confidently classified row is not lost in m + log(s) - z_y
__device__ __forceinline__ float row_nll(const float* __restrict__ z, int C, int64_t y) {
  float m = z[0];
  int am = 0;
  for (int c = 1; c < C; ++c)
    if (z[c] > m) {
      m = z[c];
      am = c;
    }
  float t = 0.f;
  for (int c = 0; c < C; ++c)
    if (c != am) t += expf(z[c] - m);
  return log1pf(t) - (z[y] - m);
}

// partial[b] = sum of the NLL of the rows of slab b (rows strided by thread inside a slab,
// combined in a fixed tree): deterministic
__global__ void __launch_bounds__(kCeThreads)
    k_ce_fwd(const float* __restrict__ logits, const int64_t* __restrict__ target, int64_t N, int C,
             int64_t rows_per_block, float* __restrict__ partial, int32_t* __restrict__ bad) {
  __shared__ float red[kCeThreads];
  const int64_t n0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t n1 = n0 + rows_per_block < N ? n0 + rows_per_block : N;
  float s = 0.f;
  for (int64_t n = n0 + threadIdx.x; n < n1; n += kCeThreads) {
    const int64_t y = target[n];
    if (y < 0 || y >= C) {   // the row's loss is NaN, so is the sum
      *bad = 1;
      s += __int_as_float(0x7fc00000);
      continue;
    }
    s += row_nll(logits + n * C, C, y);
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = kCeThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
}

__global__ void __launch_bounds__(kCeThreads)
    k_ce_finish(const float* __restrict__ partial, int P, float scale, float* __restrict__ out) {
  __shared__ float red[kCeThreads];
  float s = 0.f;
  for (int i = threadIdx.x; i < P; i += kCeThreads) s += partial[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = kCeThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0] * scale;
}

// dlogits[n,c] = (softmax(z_n)[c] - [c == y_n]) * scale * upstream[0], the label's class as -(sum of the other
// classes' exp(z_c - m)) / s (1 - p_y cancels for a confident row); a row with a label outside [0, C) is NaN
__global__ void __launch_bounds__(kCeThreads)
    k_ce_bwd(const float* __restrict__ logits, const int64_t* __restrict__ target, int64_t N, int C,
             float scale, const float* __restrict__ upstream, float* __restrict__ dlogits) {
  const float g = scale * (upstream ? upstream[0] : 1.f);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += stride) {
    const float* z = logits + n * C;
    float m = z[0];
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    const int64_t y = target[n];
    float s = 0.f, t = 0.f;
    for (int c = 0; c < C; ++c) {
      const float e = expf(z[c] - m);
      s += e;
      if (c != y) t += e;
    }
    const float inv = (y < 0 || y >= C) ? __int_as_float(0x7fc00000) : 1.f / s;
    for (int c = 0; c < C; ++c) dlogits[n * C + c] = (c == y ? -t : expf(z[c] - m)) * inv * g;
  }
}

}  // namespace mgcn

using namespace mgcn;

static int ce_blocks(int64_t N) {
  int64_t b = ceil_div(N > 0 ? N : 1, (int64_t)kCeThreads * 8);
  if (b > kNumSMs * 8) b = kNumSMs * 8;
  return (int)b;
}

extern "C" int mgcn_cross_entropy_fwd(const float* logits, const int64_t* target, int64_t N,
                                      int64_t C, int mean, float* loss, int32_t* bad_target,
                                      void* workspace, size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(N >= 0 && C >= 1 && C <= 4096, MGCN_ERR_SHAPE);
  const int P = ce_blocks(N);
  WorkspaceCarver ws(workspace);
  float* partial = ws.take<float>(P);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(loss && bad_target, MGCN_ERR_NULL);
  MGCN_REQUIRE(N == 0 || (logits && target), MGCN_ERR_NULL);
  MGCN_CHECK_CUDA(cudaMemsetAsync(bad_target, 0, sizeof(int32_t), static_cast<cudaStream_t>(stream)));
  const int64_t rows_per_block = ceil_div(N > 0 ? N : 1, P);
  MGCN_LAUNCH(k_ce_fwd, P, kCeThreads, 0, stream, logits, target, N, (int)C, rows_per_block, partial,
              bad_target);
  // the mean over no rows is NaN, as torch's
  const float scale = mean ? (N > 0 ? 1.0f / (float)N : std::numeric_limits<float>::quiet_NaN()) : 1.f;
  MGCN_LAUNCH(k_ce_finish, 1, kCeThreads, 0, stream, partial, P, scale, loss);
  return MGCN_OK;
}

extern "C" int mgcn_cross_entropy_bwd(const float* logits, const int64_t* target, int64_t N,
                                      int64_t C, int mean, const float* upstream, float* dlogits,
                                      void* stream) {
  MGCN_REQUIRE(N >= 0 && C >= 1 && C <= 4096, MGCN_ERR_SHAPE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(logits && target && dlogits, MGCN_ERR_NULL);
  const float scale = mean ? 1.0f / (float)N : 1.f;
  int64_t blocks = ceil_div(N, kCeThreads);
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  MGCN_LAUNCH(k_ce_bwd, (unsigned)blocks, kCeThreads, 0, stream, logits, target, N, (int)C, scale,
              upstream, dlogits);
  return MGCN_OK;
}

// -------------------------------------------------------------------------------------------------
// Binary-classification counters of src/gcn_meta/optim/metrics.py:8-24 (train_botnet.py:296-305) in one pass:
// counts = {TP, FP, TN, FN, correct} over pred = argmax(logits, 1) (first maximal class) or a given pred.
// The reference makes five boolean-mask passes with a host synchronisation each.  Integer sums: exact and
// independent of scheduling.
// -------------------------------------------------------------------------------------------------
namespace mgcn {
__global__ void __launch_bounds__(256)
    k_confusion(const float* __restrict__ logits, const int64_t* __restrict__ pred, int64_t N, int C,
                const int64_t* __restrict__ target, unsigned long long* __restrict__ counts) {
  unsigned long long c5[5] = {0ull, 0ull, 0ull, 0ull, 0ull};
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
    int64_t p;
    if (logits) {
      const float* z = logits + n * C;
      float m = z[0];
      p = 0;
      for (int c = 1; c < C; ++c) {
        if (z[c] > m) {
          m = z[c];
          p = c;
        }
      }
    } else {
      p = pred[n];
    }
    const int64_t y = target[n];
    c5[0] += (p == 1 && y == 1);
    c5[1] += (p == 1 && y == 0);
    c5[2] += (p == 0 && y == 0);
    c5[3] += (p == 0 && y == 1);
    c5[4] += (p == y);
  }
  __shared__ unsigned long long red[8][5];
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    unsigned long long v = c5[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    unsigned long long v = 0ull;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
    if (v) atomicAdd(counts + threadIdx.x, v);
  }
}
}  // namespace mgcn

extern "C" int mgcn_binary_confusion(const float* logits, const int64_t* pred, int64_t N, int64_t C,
                                     const int64_t* target, int64_t* counts5, void* stream) {
  MGCN_REQUIRE(counts5 != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(N >= 0 && C >= 1 && C < (int64_t(1) << 20), MGCN_ERR_RANGE);
  MGCN_REQUIRE((logits != nullptr) != (pred != nullptr) || N == 0, MGCN_ERR_NULL);   // exactly one source
  MGCN_CHECK_CUDA(cudaMemsetAsync(counts5, 0, 5 * sizeof(int64_t), static_cast<cudaStream_t>(stream)));
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(target != nullptr, MGCN_ERR_NULL);
  int64_t blocks = ceil_div(N, 256 * 4);
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  MGCN_LAUNCH(k_confusion, (unsigned)blocks, 256, 0, stream, logits, pred, N, (int)C, target,
              reinterpret_cast<unsigned long long*>(counts5));
  return MGCN_OK;
}
