// The step right behind the hot path as ONE forward and ONE backward launch (SURVEY §8 f3):
//   logits = x F^T + f                      self.final = nn.Linear(H, C)                 gcn_model.py:73,108
//   loss   = CrossEntropyLoss(logits, y)    mean or sum over the nodes                    train_botnet.py:225,287
//   TP / FP / TN / FN / correct             argmax against the labels                     train_botnet.py:296-305,
//                                                                                        optim/metrics.py:8-24
// Round 1 ran them as k_linear_small_out, k_ce_fwd, k_ce_finish (+ k_confusion) forward and k_ce_bwd,
// k_wgrad_narrow, k_reduce_partials x2, k_linear_small_in backward: five passes over [N,H] / [N,C] arrays.  Here the
// forward reads x once (writes the logits, which the caller needs anyway) and the backward reads x and the logits
// once and writes dx; loss, weight-gradient and bias-gradient sums are fixed-order two-stage reductions, the
// counters integer sums (exact): deterministic, no floating-point atomics.
//
// Thread mapping: L = H / 4 lanes own a row (one float4 each), 32 / L rows per warp; C <= kHeadMaxC classes.
#include <limits>

#include "common.cuh"

namespace mgcn {

constexpr int kHeadMaxC = 8;
constexpr int kHeadThreads = 256;

template <int L>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct HeadArgs {
  const float* x;          // [N,H]
  const float* w;          // [C,H] nn.Linear.weight
  const float* b;          // [C] or NULL
  const int64_t* target;   // [N]
  float* logits;           // [N,C]
  float* part_loss;        // [grid]
  unsigned long long* counts;   // [5] TP FP TN FN correct, or NULL
  int32_t* bad;            // [1]
  // backward
  const float* scale;      // device scalar: upstream gradient, or NULL (= 1)
  float scale_const;       // 1/N for the mean, 1 for the sum
  float* dx;               // [N,H] or NULL
  float* part_w;           // [grid][C][H]
  float* part_b;           // [grid][C]
  int64_t N;
  int C;
};

// CM = compile-time bound on the class count (2: the botnet head; 8: anything up to kHeadMaxC) — the per-class arrays
// live in registers, and at CM = 8 they cost the occupancy that hides the latency of the row loads.  Two rows per
// thread and iteration are loaded before either is used (same summation order as one row per iteration).
template <int L, int CM>
__global__ void __launch_bounds__(kHeadThreads) k_head_ce_fwd(const HeadArgs a) {
  constexpr int H = 4 * L, RPW = 32 / L;
  __shared__ float ws[kHeadMaxC][H];
  __shared__ float red[kHeadThreads / 32];
  __shared__ unsigned long long cred[kHeadThreads / 32][5];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < a.C * H; i += kHeadThreads) ws[i / H][i % H] = __ldg(a.w + i);
  __syncthreads();
  const int sub = lane % L, rw = lane / L;
  float loss = 0.f;
  unsigned long long cnt[5] = {0ull, 0ull, 0ull, 0ull, 0ull};
  float bv[CM];
#pragma unroll
  for (int c = 0; c < CM; ++c) bv[c] = (c < a.C && a.b) ? __ldg(a.b + c) : 0.f;
  const int64_t rows_per_iter = (int64_t)gridDim.x * (kHeadThreads / 32) * RPW;
  // a block owns a contiguous slab of rows (fixed summation order per block)
  const int64_t iters = (a.N + rows_per_iter - 1) / rows_per_iter;
  const int64_t slab0 = (int64_t)blockIdx.x * iters * (kHeadThreads / 32) * RPW;
  auto row_of = [&](int64_t it) { return slab0 + (it * (kHeadThreads / 32) + warp) * RPW + rw; };
  auto process = [&](int64_t n, bool ok, const float4 xv, int64_t y) {
    float z[CM];
#pragma unroll
    for (int c = 0; c < CM; ++c) {
      if (c < a.C) {
        const float4 wv = *reinterpret_cast<const float4*>(&ws[c][4 * sub]);
        float p = xv.x * wv.x;
        p = fmaf(xv.y, wv.y, p);
        p = fmaf(xv.z, wv.z, p);
        p = fmaf(xv.w, wv.w, p);
        z[c] = group_sum<L>(p) + bv[c];
      }
    }
    if (ok && sub == 0) {
      float m = z[0];
      int am = 0;
#pragma unroll
      for (int c = 1; c < CM; ++c)
        if (c < a.C && z[c] > m) {
          m = z[c];
          am = c;
        }
      // t = sum over the classes other than the argmax of exp(z_c - m); exp(z_am - m) = 1 is left out so that the
      // NLL of a confidently classified row, log1p(t) - (z_y - m), does not vanish into m + log(1 + t) - z_y
      float t = 0.f;
#pragma unroll
      for (int c = 0; c < CM; ++c)
        if (c < a.C) {
          if (c != am) t += expf(z[c] - m);
          a.logits[n * a.C + c] = z[c];
        }
      if (y < 0 || y >= a.C) {   // the row's loss is NaN, so is the sum; the counters skip it
        *a.bad = 1;
        loss += __int_as_float(0x7fc00000);
      } else {
        float zy = z[0];
#pragma unroll
        for (int c = 1; c < CM; ++c)
          if (c == (int)y) zy = z[c];
        loss += log1pf(t) - (zy - m);
        if (a.counts) {   // optim/metrics.py:8-24: positives are class 1
          cnt[0] += (am == 1 && y == 1) ? 1u : 0u;
          cnt[1] += (am == 1 && y == 0) ? 1u : 0u;
          cnt[2] += (am == 0 && y == 0) ? 1u : 0u;
          cnt[3] += (am == 0 && y == 1) ? 1u : 0u;
          cnt[4] += (am == (int)y) ? 1u : 0u;
        }
      }
    }
  };
  for (int64_t it = 0; it < iters; it += 2) {
    const int64_t n0 = row_of(it), n1 = row_of(it + 1);
    const bool ok0 = n0 < a.N, ok1 = it + 1 < iters && n1 < a.N;
    float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
    int64_t y0 = 0, y1 = 0;
    if (ok0) x0 = __ldg(reinterpret_cast<const float4*>(a.x + n0 * H) + sub);
    if (ok1) x1 = __ldg(reinterpret_cast<const float4*>(a.x + n1 * H) + sub);
    if (ok0 && sub == 0) y0 = __ldg(a.target + n0);
    if (ok1 && sub == 0) y1 = __ldg(a.target + n1);
    process(n0, ok0, x0, y0);
    process(n1, ok1, x1, y1);
  }
  // warp: lanes in a fixed butterfly; block: warps in order
  for (int o = 16; o > 0; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
  if (lane == 0) red[warp] = loss;
  if (a.counts) {
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      unsigned long long v = cnt[q];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) cred[warp][q] = v;
    }
  }
  __syncthreads();
  if (tid == 0) {
    float s = red[0];
#pragma unroll
    for (int w = 1; w < kHeadThreads / 32; ++w) s += red[w];
    a.part_loss[blockIdx.x] = s;
  }
  if (a.counts && tid < 5) {
    unsigned long long v = 0ull;
#pragma unroll
    for (int w = 0; w < kHeadThreads / 32; ++w) v += cred[w][tid];
    if (v) atomicAdd(a.counts + tid, v);   // integer sums: exact in any order
  }
}

__global__ void __launch_bounds__(256) k_head_loss_finish(const float* __restrict__ part, int P, float scale,
                                                          float* __restrict__ out) {
  __shared__ float red[256];
  float s = 0.f;
  for (int i = threadIdx.x; i < P; i += 256) s += part[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0] * scale;
}

// dl = (softmax(logits) - onehot) * g;  dx = dl F;  dF[c] += dl[c] x;  df[c] += dl[c]
template <int L, int CM>
__global__ void __launch_bounds__(kHeadThreads) k_head_ce_bwd(const HeadArgs a) {
  constexpr int H = 4 * L, RPW = 32 / L;
  __shared__ float ws[kHeadMaxC][H];
  __shared__ float redw[kHeadThreads / 32][CM][H];
  __shared__ float redb[kHeadThreads / 32][CM];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < a.C * H; i += kHeadThreads) ws[i / H][i % H] = __ldg(a.w + i);
  __syncthreads();
  const int sub = lane % L, rw = lane / L;
  const float g = a.scale_const * (a.scale ? __ldg(a.scale) : 1.f);
  float4 accw[CM];
  float accb[CM];
#pragma unroll
  for (int c = 0; c < CM; ++c) {
    accw[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    accb[c] = 0.f;
  }
  const int64_t rows_per_iter = (int64_t)gridDim.x * (kHeadThreads / 32) * RPW;
  const int64_t iters = (a.N + rows_per_iter - 1) / rows_per_iter;
  const int64_t slab0 = (int64_t)blockIdx.x * iters * (kHeadThreads / 32) * RPW;
  auto row_of = [&](int64_t it) { return slab0 + (it * (kHeadThreads / 32) + warp) * RPW + rw; };
  struct Row {
    float4 xv;
    float z[CM];
    int64_t y;
  };
  auto load = [&](int64_t n, bool ok) {
    Row r;
    r.xv = make_float4(0.f, 0.f, 0.f, 0.f);
    r.y = 0;
#pragma unroll
    for (int c = 0; c < CM; ++c) r.z[c] = 0.f;
    if (ok) {
      r.xv = __ldg(reinterpret_cast<const float4*>(a.x + n * H) + sub);
#pragma unroll
      for (int c = 0; c < CM; ++c)
        if (c < a.C) r.z[c] = __ldg(a.logits + n * a.C + c);
      r.y = __ldg(a.target + n);
    }
    return r;
  };
  auto process = [&](int64_t n, bool ok, const Row& r) {
    if (!ok) return;   // whole groups leave together
    float m = -3.4e38f;
#pragma unroll
    for (int c = 0; c < CM; ++c)
      if (c < a.C) m = fmaxf(m, r.z[c]);
    float e[CM];
    float s = 0.f, t = 0.f;   // t = sum of e_c over c != y
#pragma unroll
    for (int c = 0; c < CM; ++c)
      if (c < a.C) {
        e[c] = expf(r.z[c] - m);
        s += e[c];
        if (c != r.y) t += e[c];
      }
    // a label outside [0, C) makes the whole row NaN (and with it dw and db)
    const float inv = (r.y < 0 || r.y >= a.C) ? __int_as_float(0x7fc00000) : 1.f / s;
    float4 dxv = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < CM; ++c)
      if (c < a.C) {
        // the label's class as -(sum of the others) / s: 1 - e_y / s cancels for a confident row
        const float dl = (c == r.y ? -t : e[c]) * inv * g;
        const float4 wv = *reinterpret_cast<const float4*>(&ws[c][4 * sub]);
        dxv.x = fmaf(dl, wv.x, dxv.x);
        dxv.y = fmaf(dl, wv.y, dxv.y);
        dxv.z = fmaf(dl, wv.z, dxv.z);
        dxv.w = fmaf(dl, wv.w, dxv.w);
        accw[c].x = fmaf(dl, r.xv.x, accw[c].x);
        accw[c].y = fmaf(dl, r.xv.y, accw[c].y);
        accw[c].z = fmaf(dl, r.xv.z, accw[c].z);
        accw[c].w = fmaf(dl, r.xv.w, accw[c].w);
        if (sub == 0) accb[c] += dl;
      }
    if (a.dx) reinterpret_cast<float4*>(a.dx + n * H)[sub] = dxv;
  };
  for (int64_t it = 0; it < iters; it += 2) {
    const int64_t n0 = row_of(it), n1 = row_of(it + 1);
    const bool ok0 = n0 < a.N, ok1 = it + 1 < iters && n1 < a.N;
    const Row r0 = load(n0, ok0), r1 = load(n1, ok1);   // both rows in flight before either is used
    process(n0, ok0, r0);
    process(n1, ok1, r1);
  }
  // rows of a warp (lanes with the same sub) added in a fixed butterfly, warps in order
#pragma unroll
  for (int c = 0; c < CM; ++c) {
    if (c < a.C) {
      float4 v = accw[c];
      float bsum = accb[c];
#pragma unroll
      for (int o = L; o < 32; o <<= 1) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
        v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
        v.z += __shfl_xor_sync(0xffffffffu, v.z, o);
        v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
      }
      for (int o = 16; o > 0; o >>= 1) bsum += __shfl_xor_sync(0xffffffffu, bsum, o);
      if (rw == 0) *reinterpret_cast<float4*>(&redw[warp][c][4 * sub]) = v;
      if (lane == 0) redb[warp][c] = bsum;
    }
  }
  __syncthreads();
  for (int i = tid; i < a.C * H; i += kHeadThreads) {
    const int c = i / H, k = i % H;
    float s = redw[0][c][k];
#pragma unroll
    for (int w = 1; w < kHeadThreads / 32; ++w) s += redw[w][c][k];
    a.part_w[(int64_t)blockIdx.x * a.C * H + i] = s;
  }
  if (tid < a.C) {
    float s = redb[0][tid];
#pragma unroll
    for (int w = 1; w < kHeadThreads / 32; ++w) s += redb[w][tid];
    a.part_b[(int64_t)blockIdx.x * a.C + tid] = s;
  }
}

static int head_grid(int64_t N) {
  int64_t b = ceil_div(N > 0 ? N : 1, 2048);
  const int64_t cap = (int64_t)kNumSMs * 6;
  return (int)(b < cap ? b : cap);
}

}  // namespace mgcn

using namespace mgcn;

extern "C" int mgcn_head_cross_entropy_fwd(const float* x, int64_t N, int64_t H, const float* w, const float* b,
                                           int64_t C, const int64_t* target, int mean, float* logits, float* loss,
                                           int64_t* counts5, int32_t* bad_target, void* workspace,
                                           size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(N >= 0 && C >= 1 && C <= kHeadMaxC, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(H == 16 || H == 32 || H == 64 || H == 128, MGCN_ERR_SHAPE);
  const int P = head_grid(N);
  WorkspaceCarver ws(workspace);
  float* part = ws.take<float>(P);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(loss && bad_target && w, MGCN_ERR_NULL);
  MGCN_REQUIRE(N == 0 || (x && target && logits), MGCN_ERR_NULL);
  MGCN_REQUIRE(N == 0 || aligned16(x), MGCN_ERR_ALIGN);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MGCN_CHECK_CUDA(cudaMemsetAsync(bad_target, 0, sizeof(int32_t), st));
  if (counts5) MGCN_CHECK_CUDA(cudaMemsetAsync(counts5, 0, 5 * sizeof(int64_t), st));
  HeadArgs a{};
  a.x = x; a.w = w; a.b = b; a.target = target; a.logits = logits; a.part_loss = part;
  a.counts = reinterpret_cast<unsigned long long*>(counts5); a.bad = bad_target; a.N = N; a.C = (int)C;
  if (C <= 2) {
    switch (H) {
      case 16: MGCN_LAUNCH((k_head_ce_fwd<4, 2>), P, kHeadThreads, 0, stream, a); break;
      case 32: MGCN_LAUNCH((k_head_ce_fwd<8, 2>), P, kHeadThreads, 0, stream, a); break;
      case 64: MGCN_LAUNCH((k_head_ce_fwd<16, 2>), P, kHeadThreads, 0, stream, a); break;
      default: MGCN_LAUNCH((k_head_ce_fwd<32, 2>), P, kHeadThreads, 0, stream, a); break;
    }
  } else {
    switch (H) {
      case 16: MGCN_LAUNCH((k_head_ce_fwd<4, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
      case 32: MGCN_LAUNCH((k_head_ce_fwd<8, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
      case 64: MGCN_LAUNCH((k_head_ce_fwd<16, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
      default: MGCN_LAUNCH((k_head_ce_fwd<32, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
    }
  }
  // the mean over no rows is NaN, as torch's
  const float scale = mean ? (N > 0 ? 1.0f / (float)N : std::numeric_limits<float>::quiet_NaN()) : 1.f;
  MGCN_LAUNCH(k_head_loss_finish, 1, 256, 0, stream, part, P, scale, loss);
  return MGCN_OK;
}

extern "C" int mgcn_head_cross_entropy_bwd(const float* x, const float* logits, int64_t N, int64_t H, const float* w,
                                           int64_t C, const int64_t* target, int mean, const float* upstream,
                                           float* dx, float* dw, float* db, void* workspace,
                                           size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(N >= 0 && C >= 1 && C <= kHeadMaxC, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(H == 16 || H == 32 || H == 64 || H == 128, MGCN_ERR_SHAPE);
  const int P = head_grid(N);
  WorkspaceCarver ws(workspace);
  float* part_w = ws.take<float>((size_t)P * C * H);
  float* part_b = ws.take<float>((size_t)P * C);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(w && dw && db, MGCN_ERR_NULL);
  MGCN_REQUIRE(N == 0 || (x && logits && target), MGCN_ERR_NULL);
  MGCN_REQUIRE(N == 0 || (aligned16(x) && (!dx || aligned16(dx))), MGCN_ERR_ALIGN);
  HeadArgs a{};
  a.x = x; a.w = w; a.target = target; a.logits = const_cast<float*>(logits); a.scale = upstream;
  a.scale_const = mean ? (N > 0 ? 1.0f / (float)N : 0.f) : 1.f;
  a.dx = dx; a.part_w = part_w; a.part_b = part_b; a.N = N; a.C = (int)C;
  if (C <= 2) {
    switch (H) {
      case 16: MGCN_LAUNCH((k_head_ce_bwd<4, 2>), P, kHeadThreads, 0, stream, a); break;
      case 32: MGCN_LAUNCH((k_head_ce_bwd<8, 2>), P, kHeadThreads, 0, stream, a); break;
      case 64: MGCN_LAUNCH((k_head_ce_bwd<16, 2>), P, kHeadThreads, 0, stream, a); break;
      default: MGCN_LAUNCH((k_head_ce_bwd<32, 2>), P, kHeadThreads, 0, stream, a); break;
    }
  } else {
    switch (H) {
      case 16: MGCN_LAUNCH((k_head_ce_bwd<4, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
      case 32: MGCN_LAUNCH((k_head_ce_bwd<8, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
      case 64: MGCN_LAUNCH((k_head_ce_bwd<16, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
      default: MGCN_LAUNCH((k_head_ce_bwd<32, kHeadMaxC>), P, kHeadThreads, 0, stream, a); break;
    }
  }
  int rc = launch_reduce_partials(part_w, P, (int)(C * H), (int)H, dw, H, 1, stream);
  if (rc == MGCN_OK) rc = launch_reduce_partials(part_b, P, (int)C, (int)C, db, 0, 1, stream);
  return rc;
}
