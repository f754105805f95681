// 'max' aggregation of the primitive seam — scatter_('max', src, index, dim_size) (common.py:54-64: torch_scatter
// scatter_max with fill -1e38, untouched rows set to 0) — and of NodeModelAdditive(aggr='max')
// (gcn_base_models.py:223-237: max over the edges of (x W)[row] * norm), with the autograd of torch_scatter's
// scatter_max (the gradient of out[i,c] goes to the FIRST entry that attains the maximum).
//   forward   out[i,c] = max_k v_k * x[idx_k, c] over the row's entries in row order (= edge_index order: the
//             structure is a stable sort), arg[i,c] = edge id (perm) of the first maximal entry, -1 / 0 for an empty row;
//             with a fill value (torch_scatter's running maximum starts at fill_value and only a strictly greater entry
//             replaces it) an entry <= fill never wins, and a (row, column) without a winner is 0 / -1 as well
//   backward  primitive seam: dsrc[arg[i,c], c] = g[i,c] (an edge belongs to one row: no conflicts)
//             layer seam: a row-owned pass over the structure grouped by source,
//             dx[j,c] = sum_{k in row j} [arg[target_k, c] == edge_k] * v_k * g[target_k, c]
// Row-owned, no atomics: deterministic.  One thread per (row, column); consecutive threads take consecutive columns.
#include "common.cuh"

namespace mgcn {

// kFill: the running maximum starts at `fill` and an entry must be strictly greater to win; otherwise the row's first
// entry always wins
template <bool kFill>
__global__ void __launch_bounds__(256)
    k_segment_max(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ idx, const int32_t* __restrict__ perm,
                  const float* __restrict__ x, const float* __restrict__ edge_val, int64_t n_rows, int H, float fill,
                  float* __restrict__ out, int32_t* __restrict__ arg) {
  const int64_t total = n_rows * H;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / H;
    const int c = (int)(t - i * H);
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1);
    float best = kFill ? fill : 0.f;
    int32_t who = -1;
    for (int k = beg; k < end; ++k) {
      float v = __ldg(x + (int64_t)__ldg(idx + k) * H + c);
      if (edge_val) v = __fmul_rn(v, __ldg(edge_val + k));
      if ((!kFill && who < 0) || v > best) {
        best = v;
        who = __ldg(perm + k);
      }
    }
    out[t] = who < 0 ? 0.f : best;
    arg[t] = who;
  }
}

__global__ void __launch_bounds__(256)
    k_segment_max_bwd(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ perm,
                      const float* __restrict__ g, const int32_t* __restrict__ arg, const float* __restrict__ edge_val,
                      int64_t n_rows, int H, float* __restrict__ dx) {
  const int64_t total = n_rows * H;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = t / H;
    const int c = (int)(t - j * H);
    const int beg = __ldg(rowptr + j), end = __ldg(rowptr + j + 1);
    float s = 0.f;
    for (int k = beg; k < end; ++k) {
      const int64_t tgt = __ldg(nbr + k);
      if (__ldg(arg + tgt * H + c) == __ldg(perm + k)) {
        float v = __ldg(g + tgt * H + c);
        if (edge_val) v = __fmul_rn(v, __ldg(edge_val + k));
        s = __fadd_rn(s, v);
      }
    }
    dx[t] = s;
  }
}

__global__ void __launch_bounds__(256)
    k_scatter_max_bwd(const int32_t* __restrict__ arg, const float* __restrict__ g, int64_t total, int H, int64_t n_src,
                      float* __restrict__ dsrc) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int32_t e = arg[t];
    if (e >= 0 && e < n_src) dsrc[(int64_t)e * H + (t % H)] = g[t];
  }
}

static unsigned grid_for(int64_t total) {
  int64_t b = ceil_div(total > 0 ? total : 1, 256);
  if (b > (int64_t)kNumSMs * 16) b = (int64_t)kNumSMs * 16;
  return (unsigned)b;
}

}  // namespace mgcn

using namespace mgcn;

static int segment_max(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, int gather_perm,
                       const float* edge_val, bool with_fill, float fill, float* out, int32_t* arg, void* stream) {
  MGCN_REQUIRE(g != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H >= 1 && H <= 65536 && n_in >= 0 && g->n_rows >= 0, MGCN_ERR_SHAPE);
  if (g->n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(g->rowptr && out && arg, MGCN_ERR_NULL);
  MGCN_REQUIRE(g->nnz_cap == 0 || (g->nbr && g->perm && x), MGCN_ERR_NULL);
  const int32_t* idx = gather_perm ? g->perm : g->nbr;
  if (with_fill) {
    MGCN_LAUNCH(k_segment_max<true>, grid_for(g->n_rows * H), 256, 0, stream, g->rowptr, idx, g->perm, x, edge_val,
                g->n_rows, (int)H, fill, out, arg);
  } else {
    MGCN_LAUNCH(k_segment_max<false>, grid_for(g->n_rows * H), 256, 0, stream, g->rowptr, idx, g->perm, x, edge_val,
                g->n_rows, (int)H, 0.f, out, arg);
  }
  return MGCN_OK;
}

extern "C" int mgcn_segment_max(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, int gather_perm,
                                const float* edge_val, float* out, int32_t* arg, void* stream) {
  return segment_max(g, x, n_in, H, gather_perm, edge_val, false, 0.f, out, arg, stream);
}

extern "C" int mgcn_segment_max_ex(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, int gather_perm,
                                   const float* edge_val, float fill, float* out, int32_t* arg, void* stream) {
  return segment_max(g, x, n_in, H, gather_perm, edge_val, true, fill, out, arg, stream);
}

extern "C" int mgcn_segment_max_bwd(const mgcn_csr_t* gt, const float* grad, const int32_t* arg, const float* edge_val,
                                    int64_t H, float* dx, void* stream) {
  MGCN_REQUIRE(gt != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H >= 1 && H <= 65536 && gt->n_rows >= 0, MGCN_ERR_SHAPE);
  if (gt->n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(gt->rowptr && dx, MGCN_ERR_NULL);
  MGCN_REQUIRE(gt->nnz_cap == 0 || (gt->nbr && gt->perm && grad && arg), MGCN_ERR_NULL);
  MGCN_LAUNCH(k_segment_max_bwd, grid_for(gt->n_rows * H), 256, 0, stream, gt->rowptr, gt->nbr, gt->perm, grad, arg,
              edge_val, gt->n_rows, (int)H, dx);
  return MGCN_OK;
}

extern "C" int mgcn_scatter_max_bwd(const int32_t* arg, const float* grad, int64_t N, int64_t H, int64_t n_src,
                                    float* dsrc, void* stream) {
  MGCN_REQUIRE(N >= 0 && H >= 1 && n_src >= 0, MGCN_ERR_SHAPE);
  if (n_src > 0) {
    MGCN_REQUIRE(dsrc != nullptr, MGCN_ERR_NULL);
    MGCN_CHECK_CUDA(cudaMemsetAsync(dsrc, 0, (size_t)n_src * H * sizeof(float), static_cast<cudaStream_t>(stream)));
  }
  if (N == 0 || n_src == 0) return MGCN_OK;
  MGCN_REQUIRE(arg && grad, MGCN_ERR_NULL);
  MGCN_LAUNCH(k_scatter_max_bwd, grid_for(N * H), 256, 0, stream, arg, grad, N * H, (int)H, n_src, dsrc);
  return MGCN_OK;
}

// -------------------------------------------------------------------------------------------------
// Per-edge dot product — the gradient of an aggregation with respect to a per-edge weight
// (edge gates: gcn_base_models.py:230-232, EdgeGateProj :322-369):
//     out[e] = s_src[row_e] * s_tgt[col_e] * sum_c a[col_e, c] * b[row_e, c]
// 8 lanes per edge, fixed butterfly over the lanes: deterministic.
// -------------------------------------------------------------------------------------------------
namespace mgcn {
template <typename Index>
__global__ void __launch_bounds__(256)
    k_edge_dot(const Index* __restrict__ ei, int64_t E, const float* __restrict__ a, const float* __restrict__ b, int H,
               const float* __restrict__ s_src, const float* __restrict__ s_tgt, float* __restrict__ out) {
  const int sub = threadIdx.x & 7;
  const int64_t per_iter = (int64_t)gridDim.x * (blockDim.x >> 3);
  const int64_t n_iter = (E + per_iter - 1) / per_iter;          // uniform trip count: shuffles stay converged
  for (int64_t it = 0; it < n_iter; ++it) {
    const int64_t e = it * per_iter + (int64_t)blockIdx.x * (blockDim.x >> 3) + (threadIdx.x >> 3);
    float s = 0.f;
    int64_t r = 0, c = 0;
    if (e < E) {
      r = (int64_t)ei[e];
      c = (int64_t)ei[E + e];
      for (int k = sub; k < H; k += 8) s = fmaf(__ldg(a + c * H + k), __ldg(b + r * H + k), s);
    }
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    if (e < E && sub == 0) {
      if (s_src) s *= __ldg(s_src + r);
      if (s_tgt) s *= __ldg(s_tgt + c);
      out[e] = s;
    }
  }
}
}  // namespace mgcn

template <typename Index>
static int edge_dot(const Index* edge_index, int64_t E, const float* a, const float* b, int64_t H,
                    const float* scale_src, const float* scale_tgt, float* out, void* stream) {
  MGCN_REQUIRE(E >= 0 && H >= 1 && H <= 65536, MGCN_ERR_SHAPE);
  if (E == 0) return MGCN_OK;
  MGCN_REQUIRE(edge_index && a && b && out, MGCN_ERR_NULL);
  int64_t blocks = ceil_div(E, 32);
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  MGCN_LAUNCH(k_edge_dot<Index>, (unsigned)blocks, 256, 0, stream, edge_index, E, a, b, (int)H, scale_src, scale_tgt,
              out);
  return MGCN_OK;
}

extern "C" int mgcn_edge_dot(const int64_t* edge_index, int64_t E, const float* a, const float* b, int64_t H,
                             const float* scale_src, const float* scale_tgt, float* out, void* stream) {
  return edge_dot(edge_index, E, a, b, H, scale_src, scale_tgt, out, stream);
}

extern "C" int mgcn_edge_dot_i32(const int32_t* edge_index, int64_t E, const float* a, const float* b, int64_t H,
                                 const float* scale_src, const float* scale_tgt, float* out, void* stream) {
  return edge_dot(edge_index, E, a, b, H, scale_src, scale_tgt, out, stream);
}
