// Edge gates of the hidden-32 residual stack (EdgeGateProj, gcn_base_models.py:322-369, in_edgedim None):
//
//     g_ij = sigmoid(a_j + (b_i + c)),   a_j = (x_j W) . u,   b_i = (x_i W) . v        (edge j -> i)
//
// A gate depends on the two endpoints of its edge only, so every kernel forms it from two per-node scores while it
// gathers (gather.cuh: edge_gate): no [E] gate array, no edge ids, duplicate edges get equal gates, and a symmetric
// structure still serves both directions.  The forward gate sits in the gather of k_gcn_fwd_tc<0, true>
// (gcn_fwd_tc.cu); this file holds the scores, the gated narrow aggregation of the first layer, and the two backward
// passes:
//
//   by target (structure of the forward)   dt_ij = <gs_i, m_j> g_ij (1 - g_ij),  db_i = sum_j dt_ij
//   by source (transposed structure)       the same dt_ij, bit for bit (same operands, same operations, same lane
//                                          layout), da_j = sum_i dt_ij,  dxw_j = pre_j sum_i g_ij gs_i + da_j u + db_j v
//
// Both passes walk the work order of their structure (mgcn_csr_t::tasks) with one 4-lane group per task (8 columns per
// lane, as gather.cuh); hub segments store partials that one more launch adds in a fixed order.  No atomics.
#include "common.cuh"
#include "gather.cuh"

namespace mgcn {

constexpr int kGpWarps = 8;

// ---- scores --------------------------------------------------------------------------------------
// narrow inputs (H <= 4, the first layer): a thread per row
__global__ void __launch_bounds__(256) k_gate_scores(const float* __restrict__ x, int64_t N, int H,
                                                     const float* __restrict__ in_scale, const float* __restrict__ w,
                                                     const float* __restrict__ u, const float* __restrict__ v,
                                                     float2* __restrict__ ab) {
  __shared__ float wu[32], wv[32];
  if (threadIdx.x < H) {
    const int k = threadIdx.x;
    float su = 0.f, sv = 0.f;
    for (int n = 0; n < 32; ++n) {
      su = __fmaf_rn(__ldg(w + k * 32 + n), __ldg(u + n), su);
      sv = __fmaf_rn(__ldg(w + k * 32 + n), __ldg(v + n), sv);
    }
    wu[k] = su;
    wv[k] = sv;
  }
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    const float* xr = x + i * H;
    float sa = 0.f, sb = 0.f;
    for (int k = 0; k < H; ++k) {
      const float xv = __ldg(xr + k);
      sa = __fmaf_rn(xv, wu[k], sa);
      sb = __fmaf_rn(xv, wv[k], sb);
    }
    if (in_scale) {
      const float r = __frcp_rn(__ldg(in_scale + i));
      sa = __fmul_rn(sa, r);
      sb = __fmul_rn(sb, r);
    }
    ab[i] = make_float2(sa, sb);
  }
}

// H = 32 (the stored z of the hidden layers): a 4-lane group per row, 8 columns per lane as two 16-byte loads, the
// partial dots added by two butterfly steps (a warp load instruction covers 8 whole rows)
__global__ void __launch_bounds__(256) k_gate_scores32(const float* __restrict__ x, int64_t N,
                                                       const float* __restrict__ in_scale, const float* __restrict__ w,
                                                       const float* __restrict__ u, const float* __restrict__ v,
                                                       float2* __restrict__ ab) {
  __shared__ float wu[32], wv[32];
  if (threadIdx.x < 32) {
    const int k = threadIdx.x;
    float su = 0.f, sv = 0.f;
    for (int n = 0; n < 32; ++n) {
      su = __fmaf_rn(__ldg(w + k * 32 + n), __ldg(u + n), su);
      sv = __fmaf_rn(__ldg(w + k * 32 + n), __ldg(v + n), sv);
    }
    wu[k] = su;
    wv[k] = sv;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, sub = lane & 3, col = sub * 8;
  const unsigned gmask = 0xfu << (lane & ~3);
  const int64_t groups = ((int64_t)gridDim.x * blockDim.x) >> 2;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2; i < N; i += groups) {
    const float4 lo = __ldg(reinterpret_cast<const float4*>(x + i * 32 + col));
    const float4 hi = __ldg(reinterpret_cast<const float4*>(x + i * 32 + col + 4));
    const float e[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      sa = __fmaf_rn(e[k], wu[col + k], sa);
      sb = __fmaf_rn(e[k], wv[col + k], sb);
    }
    sa = __fadd_rn(sa, __shfl_xor_sync(gmask, sa, 1));
    sb = __fadd_rn(sb, __shfl_xor_sync(gmask, sb, 1));
    sa = __fadd_rn(sa, __shfl_xor_sync(gmask, sa, 2));
    sb = __fadd_rn(sb, __shfl_xor_sync(gmask, sb, 2));
    if (sub == 0) {
      if (in_scale) {
        const float r = __frcp_rn(__ldg(in_scale + i));
        sa = __fmul_rn(sa, r);
        sb = __fmul_rn(sb, r);
      }
      ab[i] = make_float2(sa, sb);
    }
  }
}

// ---- gated aggregation of a narrow input (H <= 4) ---------------------------------------------------
__global__ void __launch_bounds__(256) k_gate_spmm_narrow(const int32_t* __restrict__ rowptr,
                                                          const int32_t* __restrict__ nbr, int64_t n_rows, int H,
                                                          const float* __restrict__ x, const float2* __restrict__ ab,
                                                          const float* __restrict__ c, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const float gc = c ? __ldg(c) : 0.f;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_rows;
       i += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1);
    const float t = __fadd_rn(__ldg(&ab[i].y), gc);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int e = beg + lane; e < end; e += 32) {
      const int j = __ldg(nbr + e);
      const float g = edge_gate(__ldg(&ab[j].x), t);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (k < H) acc[k] = __fadd_rn(acc[k], __fmul_rn(g, __ldg(x + (int64_t)j * H + k)));
    }
    // butterfly: every lane ends with the same bits (each step adds two values, a + b == b + a)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[k] = __fadd_rn(acc[k], __shfl_xor_sync(0xffffffffu, acc[k], o));
    }
    if (lane < H) {
      float r = acc[0];
#pragma unroll
      for (int k = 1; k < 4; ++k)
        if (lane == k) r = acc[k];
      out[i * H + lane] = r;
    }
  }
}

// ---- backward passes ---------------------------------------------------------------------------------
struct GatePassArgs {
  const int4* tasks;
  const int32_t* nbr_w;
  const int32_t* seg_count;
  const int32_t* hub_rows;
  const int32_t* hub_seg0;
  const int32_t* hub_count;
  const int32_t* rowptr;
  const float* own;      // row-local operand: gs (by target) / m (by source)
  const float* gat;      // gathered operand:  m (by target) / gs (by source)
  const float2* ab;
  const float* c;
  const float* db;       // by source: db_j of the by-target pass
  const float* pre;      // by source: [N] or NULL
  const float* u;        // by source: [32]
  const float* v;        // by source: [32]
  const float* sigma;    // by source: [N] or NULL
  float* out_s;          // by target: db [N]
  float* dxw;            // by source: [N,32]
  float* dsc;            // by source: [N,3]
  float* part_s;         // [seg_cap]
  float* part_row;       // by source: [seg_cap,32]
  int64_t n_rows;
  int64_t seg_cap;
  int64_t hub_cap;
  int hub_threshold;
};

__device__ __forceinline__ Row8 ld_row8_plain(const float* p) {
  Row8 r;
  const float4 lo = __ldg(reinterpret_cast<const float4*>(p)), hi = __ldg(reinterpret_cast<const float4*>(p + 4));
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}

// <p, q> over the 32 columns of a 4-lane group: 8 fused products per lane in column order, then two butterfly steps.
// Symmetric in its operands bit for bit (fma(a, b, s) == fma(b, a, s)), and every lane of the group gets the same sum.
__device__ __forceinline__ float group_dot(const Row8& p, const Row8& q, unsigned gmask) {
  float s = __fmul_rn(p.v[0], q.v[0]);
#pragma unroll
  for (int k = 1; k < 8; ++k) s = __fmaf_rn(p.v[k], q.v[k], s);
  s = __fadd_rn(s, __shfl_xor_sync(gmask, s, 1));
  s = __fadd_rn(s, __shfl_xor_sync(gmask, s, 2));
  return s;
}

__device__ __forceinline__ float gate_dt(float dot, float g) {
  return __fmul_rn(dot, __fmul_rn(g, __fsub_rn(1.f, g)));
}

// the finished row of the by-source pass
__device__ __forceinline__ void by_source_finish(const GatePassArgs& a, int64_t row, int sub, int col, const Row8& acc,
                                                 float da) {
  const float dbj = __ldg(a.db + row);
  const float prej = a.pre ? __ldg(a.pre + row) : 1.f;
  float o[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    float r = a.pre ? __fmul_rn(prej, acc.v[q]) : acc.v[q];
    r = __fadd_rn(r, __fmul_rn(da, __ldg(a.u + col + q)));
    o[q] = __fadd_rn(r, __fmul_rn(dbj, __ldg(a.v + col + q)));
  }
  float* d = a.dxw + row * kGH + col;
  *reinterpret_cast<float4*>(d) = make_float4(o[0], o[1], o[2], o[3]);
  *reinterpret_cast<float4*>(d + 4) = make_float4(o[4], o[5], o[6], o[7]);
  if (sub == 0) {
    const float inv = a.sigma ? __frcp_rn(__ldg(a.sigma + row)) : 1.f;
    a.dsc[row * 3 + 0] = __fmul_rn(da, inv);
    a.dsc[row * 3 + 1] = __fmul_rn(dbj, inv);
    a.dsc[row * 3 + 2] = dbj;
  }
}

template <bool kBySource>
__global__ void __launch_bounds__(kGpWarps * 32) k_gate_pass(const GatePassArgs a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & 3, grp = lane >> 2, grp_lane0 = grp * 4, col = sub * 8;
  const unsigned gmask = 0xfu << grp_lane0;
  int64_t nseg = 0;
  if (a.seg_count) {
    nseg = *a.seg_count;
    if (nseg > a.seg_cap) nseg = a.seg_cap;
  }
  const int64_t limit = a.n_rows + nseg;
  const float gc = a.c ? __ldg(a.c) : 0.f;
  const int64_t stride = (int64_t)gridDim.x * kGpWarps * 8;
  for (int64_t task = ((int64_t)blockIdx.x * kGpWarps + warp) * 8 + grp; task < limit; task += stride) {
    const int4 d = __ldg(a.tasks + task);
    const int row = d.x, beg = d.y, end = d.z, slot = d.w;
    if (row < 0) continue;
    const Row8 own = ld_row8_plain(a.own + (int64_t)row * kGH + col);
    const float2 sown = __ldg(a.ab + row);
    const float t_own = __fadd_rn(sown.y, gc);   // by target: b_i + c
    Row8 acc;
#pragma unroll
    for (int q = 0; q < 8; ++q) acc.v[q] = 0.f;
    float s = 0.f;
    for (int e = beg; e < end; e += 4) {
      const int cnt = min(4, end - e);
      const int idx = (e + sub < end) ? __ldg(a.nbr_w + e + sub) : 0;
      int j[4];
      Row8 gr[4];
      float2 sj[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        j[t] = __shfl_sync(gmask, idx, grp_lane0 + t);
        if (t < cnt) {
          gr[t] = ld_row8(a.gat + (int64_t)j[t] * kGH + col);
          sj[t] = __ldg(a.ab + j[t]);
        }
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        if (t < cnt) {
          const float g = kBySource ? edge_gate(sown.x, __fadd_rn(sj[t].y, gc)) : edge_gate(sj[t].x, t_own);
          const float dt = gate_dt(group_dot(own, gr[t], gmask), g);
          s = __fadd_rn(s, dt);
          if (kBySource) {
#pragma unroll
            for (int q = 0; q < 8; ++q) acc.v[q] = __fadd_rn(acc.v[q], __fmul_rn(g, gr[t].v[q]));
          }
        }
      }
    }
    if (slot != 0) {
      if (sub == 0) a.part_s[slot - 1] = s;
      if (kBySource) store_partial(a.part_row, slot, col, acc);
    } else if (kBySource) {
      by_source_finish(a, row, sub, col, acc, s);
    } else if (sub == 0) {
      a.out_s[row] = s;
    }
  }
}

// hub rows: one warp per row, the 8 lane groups sum 8 contiguous runs of its segment partials, the run sums added left
// to right (the order of k_agg_flat_hub_finish)
template <bool kBySource>
__global__ void __launch_bounds__(256) k_gate_hub_finish(const GatePassArgs a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane & 3, grp = lane >> 2, col = sub * 8;
  int64_t nh = *a.hub_count;
  if (nh > a.hub_cap) nh = a.hub_cap;
  for (int64_t k = (int64_t)blockIdx.x * 8 + warp; k < nh; k += (int64_t)gridDim.x * 8) {
    const int64_t row = __ldg(a.hub_rows + k);
    const int s0 = __ldg(a.hub_seg0 + k);
    const int len = __ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row);
    const int ns = (len + a.hub_threshold - 1) / a.hub_threshold;
    const int per = (ns + 7) >> 3;
    const int q0 = grp * per, q1 = min(ns, q0 + per);
    float rs = 0.f;
    for (int q = q0; q < q1; ++q) rs = __fadd_rn(rs, a.part_s[s0 + q]);
    float ts = __shfl_sync(0xffffffffu, rs, 0);
    for (int g = 1; g < 8; ++g) {
      const float o = __shfl_sync(0xffffffffu, rs, 4 * g);
      if (g * per < ns) ts = __fadd_rn(ts, o);
    }
    if (kBySource) {
      const Row8 run = hub_run_sum(a.part_row, s0, q0, q1, col);
      Row8 tot;
#pragma unroll
      for (int q = 0; q < 8; ++q) tot.v[q] = __shfl_sync(0xffffffffu, run.v[q], sub);
#pragma unroll
      for (int g = 1; g < 8; ++g) {
        Row8 other;
#pragma unroll
        for (int q = 0; q < 8; ++q) other.v[q] = __shfl_sync(0xffffffffu, run.v[q], 4 * g + sub);
        if (g * per < ns) row8_add(tot, other);
      }
      if (grp == 0) by_source_finish(a, row, sub, col, tot, ts);
    } else if (lane == 0) {
      a.out_s[row] = ts;
    }
  }
}

template <bool kBySource>
int launch_gate_pass(const mgcn_csr_t* g, GatePassArgs& a, void* workspace, size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr && g != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(g->n_rows >= 0, MGCN_ERR_RANGE);
  const bool hubs = g->hub_rows && g->hub_seg0 && g->hub_count && g->seg_count && g->hub_cap > 0 && g->seg_cap > 0;
  WorkspaceCarver ws(workspace);
  a.part_s = ws.take<float>(hubs ? (size_t)g->seg_cap : 0);
  a.part_row = ws.take<float>(hubs && kBySource ? (size_t)g->seg_cap * kGH : 0);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  if (g->n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(a.own && a.gat && a.ab && g->rowptr && g->tasks, MGCN_ERR_NULL);
  MGCN_REQUIRE(g->nnz_cap == 0 || g->nbr_w, MGCN_ERR_NULL);
  MGCN_REQUIRE((reinterpret_cast<uintptr_t>(a.gat) & 31u) == 0, MGCN_ERR_ALIGN);   // 256-bit row gathers
  MGCN_REQUIRE(aligned16(a.own) && aligned16(g->tasks) && aligned16(a.part_row) && (reinterpret_cast<uintptr_t>(a.ab) & 7u) == 0,
               MGCN_ERR_ALIGN);
  a.tasks = reinterpret_cast<const int4*>(g->tasks);
  a.nbr_w = g->nbr_w;
  a.seg_count = hubs ? g->seg_count : nullptr;
  a.hub_rows = g->hub_rows;
  a.hub_seg0 = g->hub_seg0;
  a.hub_count = g->hub_count;
  a.rowptr = g->rowptr;
  a.n_rows = g->n_rows;
  a.seg_cap = hubs ? g->seg_cap : 0;
  a.hub_cap = hubs ? g->hub_cap : 0;
  a.hub_threshold = g->hub_threshold;
  int64_t blocks = ceil_div(a.n_rows + a.seg_cap, (int64_t)kGpWarps * 8);
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  MGCN_LAUNCH(k_gate_pass<kBySource>, (unsigned)blocks, kGpWarps * 32, 0, stream, a);
  if (hubs) {
    int64_t hb = ceil_div(a.hub_cap, (int64_t)8);
    if (hb > (int64_t)kNumSMs * 8) hb = (int64_t)kNumSMs * 8;
    MGCN_LAUNCH(k_gate_hub_finish<kBySource>, (unsigned)hb, 256, 0, stream, a);
  }
  return MGCN_OK;
}

}  // namespace mgcn

using namespace mgcn;

extern "C" int mgcn_gate_scores(const float* x, int64_t N, int64_t H, const float* in_scale, const float* w,
                                const float* u, const float* v, float* ab, void* stream) {
  MGCN_REQUIRE(N >= 0, MGCN_ERR_RANGE);
  MGCN_REQUIRE(H >= 1 && H <= 32, MGCN_ERR_SHAPE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(x && w && u && v && ab, MGCN_ERR_NULL);
  if (H == 32 && aligned16(x)) {
    int64_t blocks = ceil_div(N, (int64_t)64);
    if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
    MGCN_LAUNCH(k_gate_scores32, (unsigned)blocks, 256, 0, stream, x, N, in_scale, w, u, v,
                reinterpret_cast<float2*>(ab));
    return MGCN_OK;
  }
  int64_t blocks = ceil_div(N, (int64_t)256);
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  MGCN_LAUNCH(k_gate_scores, (unsigned)blocks, 256, 0, stream, x, N, (int)H, in_scale, w, u, v,
              reinterpret_cast<float2*>(ab));
  return MGCN_OK;
}

extern "C" int mgcn_gate_spmm_narrow(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, const float* ab,
                                     const float* c, float* out, void* stream) {
  MGCN_REQUIRE(g != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H >= 1 && H <= 4, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(n_in >= 0 && g->n_rows >= 0, MGCN_ERR_RANGE);
  if (g->n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(x && ab && out && g->rowptr && (g->nnz_cap == 0 || g->nbr), MGCN_ERR_NULL);
  int64_t blocks = ceil_div(g->n_rows, (int64_t)8);
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  MGCN_LAUNCH(k_gate_spmm_narrow, (unsigned)blocks, 256, 0, stream, g->rowptr, g->nbr, g->n_rows, (int)H, x,
              reinterpret_cast<const float2*>(ab), c, out);
  return MGCN_OK;
}

extern "C" int mgcn_gate_grad_by_target(const mgcn_csr_t* g, const float* gs, const float* m, const float* ab,
                                        const float* c, float* db, void* workspace, size_t* workspace_bytes,
                                        void* stream) {
  GatePassArgs a{};
  a.own = gs; a.gat = m; a.ab = reinterpret_cast<const float2*>(ab); a.c = c; a.out_s = db;
  if (workspace != nullptr && g != nullptr && g->n_rows > 0) MGCN_REQUIRE(db != nullptr, MGCN_ERR_NULL);
  return launch_gate_pass<false>(g, a, workspace, workspace_bytes, stream);
}

extern "C" int mgcn_gate_grad_by_source(const mgcn_csr_t* gt, const float* gs, const float* m, const float* ab,
                                        const float* c, const float* db, const float* pre, const float* u,
                                        const float* v, const float* sigma, float* dxw, float* dsc, void* workspace,
                                        size_t* workspace_bytes, void* stream) {
  GatePassArgs a{};
  a.own = m; a.gat = gs; a.ab = reinterpret_cast<const float2*>(ab); a.c = c;
  a.db = db; a.pre = pre; a.u = u; a.v = v; a.sigma = sigma; a.dxw = dxw; a.dsc = dsc;
  if (workspace != nullptr && gt != nullptr && gt->n_rows > 0) {
    MGCN_REQUIRE(db && u && v && dxw && dsc, MGCN_ERR_NULL);
    MGCN_REQUIRE(aligned16(dxw), MGCN_ERR_ALIGN);
  }
  return launch_gate_pass<true>(gt, a, workspace, workspace_bytes, stream);
}
