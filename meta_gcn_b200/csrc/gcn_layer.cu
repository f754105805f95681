// One residual GCN layer of the botnet model (gcn_model.py:89-106 around
// NodeModelAdditive.forward, gcn_base_models.py:199-243) at hidden = 32, as three kernels:
//
//   k_layer_fwd   (forward, one launch per layer)
//       h_i     = relu( post_i * sum_{e: col[e]=i} m[row[e]] + bias )          m = pre * (x W_n), written by
//       y_i     = h_i + x_i R_n^T + r_n                                       the previous layer's launch
//       x'_i    = act(y_i)                     -> x_next      (act = ReLU, identity for the last layer)
//       m'_i    = pre_i * (x'_i W_{n+1})       -> m_next      (messages of the next layer)
//       bits_i  = (h_i > 0) as one 32-bit word -> hmask       (all the backward needs of h)
//     A lane group of 8 lanes owns a row (float4 per lane) and sums its entries in edge_index order —
//     the reference's CPU scatter_add order — 4 rows per warp at a time, 16 rows per tile; the tile's
//     two dense products run on the tensor pipe (mma.sync m16n8k8, 3xTF32) out of shared memory, so
//     per layer the forward reads m (gathered) and x once and writes x' and m' once.
//   k_agg_plain   (agg_pipelined.cu; backward, transposed aggregation)   dxw = pre * A^T gs
//   k_layer_bwd   (backward, row-local):
//       G       = dxw W_n^T + gy R_n;   dW_n = x_n^T dxw;   dR_n = gy^T x_n;   dr_n = colsum(gy)
//       gy_prev = G * (x_n > 0);        gs_prev = post * gy_prev * bits_{n-1}
//     gy is the gradient w.r.t. y_n (outer ReLU already applied), gs the operand of the transposed
//     aggregation of layer n-1.  Weight gradients accumulate in registers over all tiles of a warp and
//     are reduced warp -> CTA -> grid in a fixed order (deterministic, no atomics).
//
// Why the tensor pipe at H = 32: 6 products of [N,32]x[32,32] per layer are 0.53 TFLOP per step at the
// botnet batch; the FP32 FMA peak (74 TFLOP/s) alone would cost 7 ms against a 5 ms HBM bound for the
// whole step (measured: FMA transforms 0.28-0.54 ms per product, scripts/microbench.py).  fp32 parity
// (rtol 1e-5) rules out single-pass TF32, hence the hi/lo split of mma_tile.cuh.
#include <cstdlib>
#include <mutex>

#include "common.cuh"
#include "gather.cuh"
#include "mma_tile.cuh"

namespace mgcn {

constexpr int kH = 32;
constexpr int kLda = kH + 4;   // activation tiles: conflict-free row-major A fragments
constexpr int kLdb = kH + 8;   // weight planes: conflict-free B fragments
constexpr int kPlane = kH * kLdb;

__device__ __forceinline__ float4 f4_add2(float4 a, float4 b) {
  // two packed f32x2 adds (sm_100 FADD2): same IEEE result per element as four scalar adds
  float4 r;
  asm("{\n .reg .b64 a0, a1, b0, b1;\n mov.b64 a0, {%4, %5};\n mov.b64 a1, {%6, %7};\n"
      " mov.b64 b0, {%8, %9};\n mov.b64 b1, {%10, %11};\n add.rn.f32x2 a0, a0, b0;\n"
      " add.rn.f32x2 a1, a1, b1;\n mov.b64 {%0, %1}, a0;\n mov.b64 {%2, %3}, a1;\n}\n"
      : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
      : "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w));
  return r;
}

__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;\n" ::: "memory");
}

// plane(k, c) = w[k*stride_k + c*stride_c] split into tf32 hi / lo, [kH][kLdb] each
__device__ __forceinline__ void fill_plane(const float* __restrict__ w, int stride_k, int stride_c,
                                           float* __restrict__ hi, float* __restrict__ lo, int tid,
                                           int nthreads) {
  for (int i = tid; i < kH * kH; i += nthreads) {
    const int k = i / kH, c = i % kH;
    uint32_t h, l;
    split_tf32(__ldg(w + k * stride_k + c * stride_c), h, l);
    hi[k * kLdb + c] = __uint_as_float(h);
    lo[k * kLdb + c] = __uint_as_float(l);
  }
}

struct LayerFwdArgs {
  const int4* tasks;        // work descriptors (mgcn_csr_t::tasks)
  const int32_t* nbr_w;     // index stream in work order (mgcn_csr_t::nbr_w)
  const int32_t* seg_count;
  const int32_t* hub_rows;
  const int32_t* hub_seg0;
  const int32_t* hub_count;
  const int32_t* rowptr;
  const float* m;           // [n_in, 32] messages, pre-scaled by the per-source factor
  const float* x;           // [N, 32] layer input (residual operand), or NULL when resid is given
  const float* resid;       // [N, 32] finished residual term x R^T + r (first layer, H_in != 32)
  const float* res_w;       // [32][32] nn.Linear.weight (out, in)
  const float* res_b;       // [32] or NULL
  const float* w_next;      // [32][32] weight_node of the next layer (in, out), or NULL
  const float* bias;        // node-model bias [32] or NULL
  const float* pre;         // per-source factor of the NEXT layer's messages, or NULL
  const float* post;        // per-target factor, or NULL
  const float* out_scale;   // [N] or NULL: x_next rows leave multiplied by it (the aggregate-then-transform stack stores
                            // its activations with the per-source factor applied, csrc/gcn_fwd_tc.cu)
  // first layer with a narrow input (row-local mode only): z = npost * (ns W_in), resid = nx R^T + r, formed
  // in the kernel from [N, nhin] operands instead of being read as two [N, 32] arrays
  const float* ns;          // [N, nhin]  aggregated narrow input  sum_j pre_j x_j
  const float* nx;          // [N, nhin]  narrow layer input
  const float* nw;          // [nhin][32] weight_node of the first layer (in, out)
  const float* npost;       // [N] per-target factor or NULL
  int nhin;
  const uint32_t* keep;     // [N] dropout keep bits (streaming first layer only), or NULL
  float keep_scale;         // 1 / (1 - p)
  float* x_next;            // [N, 32]
  float* m_next;            // [N, 32] (with w_next)
  uint32_t* hmask;          // [N]
  float* partial;           // [seg_cap, 32] hub segment sums
  int64_t n_rows;
  int64_t seg_cap;
  int64_t hub_cap;
  int act_out;
  int hub_threshold;
};

#ifndef MGCN_FWD_MINB
#define MGCN_FWD_MINB 5   // resident CTAs per SM the forward kernel is compiled for
#endif
#ifndef MGCN_AGG_MINB
#define MGCN_AGG_MINB 3
#endif
#ifndef MGCN_AGG_WARPS
#define MGCN_AGG_WARPS 8   // warps per CTA of the plain aggregation
#endif

// Descriptors of a 16-task tile: lanes 0..15 load one each (empty task past `limit`).
__device__ __forceinline__ int4 load_tile_desc(const int4* __restrict__ tasks, int64_t base, int64_t limit,
                                               int lane, uint64_t pol) {
  int4 d = make_int4(-1, 0, 0, 0);
  if (lane < 16 && base + lane < limit) d = ld_i4_hint(tasks + base + lane, pol);
  return d;
}

// h = relu(post * acc + bias) -> Hs row, mask word -> hmask[row]
__device__ __forceinline__ void finish_h(const LayerFwdArgs& a, Row8 acc, float post, int64_t row,
                                         float* __restrict__ hs_row, int sub, unsigned gmask, int col) {
  if (a.post) {
#pragma unroll
    for (int q = 0; q < 8; ++q) acc.v[q] = __fmul_rn(acc.v[q], post);
  }
  if (a.bias) {
#pragma unroll
    for (int q = 0; q < 8; ++q) acc.v[q] = __fadd_rn(acc.v[q], __ldg(a.bias + col + q));
  }
  uint32_t bits = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    acc.v[q] = acc.v[q] > 0.f ? acc.v[q] : 0.f;
    bits |= (acc.v[q] > 0.f ? 1u : 0u) << q;
  }
  *reinterpret_cast<float4*>(hs_row + col) = make_float4(acc.v[0], acc.v[1], acc.v[2], acc.v[3]);
  *reinterpret_cast<float4*>(hs_row + col + 4) = make_float4(acc.v[4], acc.v[5], acc.v[6], acc.v[7]);
  bits <<= col;
  bits |= __shfl_xor_sync(gmask, bits, 1);
  bits |= __shfl_xor_sync(gmask, bits, 2);
  if (sub == 0) a.hmask[row] = bits;
}

constexpr int kGiantSegs = 32;   // hubs with more segments are summed by a whole CTA (64 runs) instead of a warp (8 runs)
constexpr int kGiantList = 32;

__global__ void __launch_bounds__(256) k_hub_reduce(const int32_t* __restrict__ hub_rows,
                                                    const int32_t* __restrict__ hub_seg0,
                                                    const int32_t* __restrict__ hub_count,
                                                    const int32_t* __restrict__ rowptr, int64_t hub_cap,
                                                    int hub_threshold, float* __restrict__ partial) {
  __shared__ int giant_k[kGiantList];
  __shared__ int n_giant;
  __shared__ __align__(16) float red[64][kH];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane & 3, grp = lane >> 2, col = sub * 8;
  int64_t nh = *hub_count;
  if (nh > hub_cap) nh = hub_cap;
  const int64_t W = (int64_t)gridDim.x * 8;
  int64_t k = (int64_t)blockIdx.x * 8 + warp;
  // rounds: a warp that finds the giant list full stops at that hub and resumes there after the list is drained, so
  // every giant gets the 64-run grouping whatever the grid (and hence the device's SM count) and the hub table order
  bool more = true;
  while (more) {
    if (threadIdx.x == 0) n_giant = 0;
    __syncthreads();
    for (; k < nh; k += W) {
      const int64_t row = __ldg(hub_rows + k);
      const int s0 = __ldg(hub_seg0 + k);
      const int len = __ldg(rowptr + row + 1) - __ldg(rowptr + row);
      const int ns = (len + hub_threshold - 1) / hub_threshold;
      if (ns <= 1) continue;
      if (ns > kGiantSegs) {   // queue for the CTA-wide pass below (the slot order never reaches the results)
        int slot = 0;
        if (lane == 0) slot = atomicAdd(&n_giant, 1);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot >= kGiantList) break;   // list full: this hub waits for the next round
        if (lane == 0) giant_k[slot] = (int)k;
        continue;
      }
      const int per = (ns + 7) >> 3;
      const Row8 run = hub_run_sum(partial, s0, grp * per, min(ns, grp * per + per), col);
      Row8 tot = run;   // group 0: its own run; then runs 1..7 in order
#pragma unroll
      for (int g = 1; g < 8; ++g) {
        Row8 other;
#pragma unroll
        for (int q = 0; q < 8; ++q) other.v[q] = __shfl_sync(0xffffffffu, run.v[q], 4 * g + sub);
        if (g * per < ns) row8_add(tot, other);
      }
      if (grp == 0) {
        float* o = partial + (int64_t)s0 * kH + col;
        *reinterpret_cast<float4*>(o) = make_float4(tot.v[0], tot.v[1], tot.v[2], tot.v[3]);
        *reinterpret_cast<float4*>(o + 4) = make_float4(tot.v[4], tot.v[5], tot.v[6], tot.v[7]);
      }
    }
    __syncthreads();
    // giants: 64 lane groups of the CTA sum 64 contiguous runs concurrently, group 0 adds the 64 run sums in order
    const int ng = min(n_giant, kGiantList);
    for (int gi = 0; gi < ng; ++gi) {
      const int64_t k = giant_k[gi];
      const int64_t row = __ldg(hub_rows + k);
      const int s0 = __ldg(hub_seg0 + k);
      const int len = __ldg(rowptr + row + 1) - __ldg(rowptr + row);
      const int ns = (len + hub_threshold - 1) / hub_threshold;
      const int per = (ns + 63) >> 6, gid = warp * 8 + grp;
      const Row8 run = hub_run_sum(partial, s0, gid * per, min(ns, gid * per + per), col);
      *reinterpret_cast<float4*>(&red[gid][col]) = make_float4(run.v[0], run.v[1], run.v[2], run.v[3]);
      *reinterpret_cast<float4*>(&red[gid][col + 4]) = make_float4(run.v[4], run.v[5], run.v[6], run.v[7]);
      __syncthreads();   // also: every read of the hub's first slot (run 0) has completed
      if (warp == 0 && grp == 0) {
        Row8 tot = run;
        for (int g = 1; g < 64 && g * per < ns; ++g) {
          const float4 lo = *reinterpret_cast<const float4*>(&red[g][col]), hi = *reinterpret_cast<const float4*>(&red[g][col + 4]);
          Row8 o;
          o.v[0] = lo.x; o.v[1] = lo.y; o.v[2] = lo.z; o.v[3] = lo.w;
          o.v[4] = hi.x; o.v[5] = hi.y; o.v[6] = hi.z; o.v[7] = hi.w;
          row8_add(tot, o);
        }
        float* o = partial + (int64_t)s0 * kH + col;
        *reinterpret_cast<float4*>(o) = make_float4(tot.v[0], tot.v[1], tot.v[2], tot.v[3]);
        *reinterpret_cast<float4*>(o + 4) = make_float4(tot.v[4], tot.v[5], tot.v[6], tot.v[7]);
      }
      __syncthreads();
    }
    more = __syncthreads_or(k < nh) != 0;   // also: n_giant is read above by every thread before it is reset
  }
}

static inline int launch_hub_reduce(const mgcn_csr_t* g, float* partial, void* stream) {
  int64_t hb = ceil_div(g->hub_cap, 8);
  if (hb > (int64_t)kNumSMs * 8) hb = (int64_t)kNumSMs * 8;
  MGCN_LAUNCH(k_hub_reduce, (unsigned)hb, 256, 0, stream, g->hub_rows, g->hub_seg0, g->hub_count, g->rowptr,
              g->hub_cap, g->hub_threshold, partial);
  return MGCN_OK;
}

// residual operand rows (x, or the finished residual term) of a 16-row tile -> Xs, asynchronously
__device__ __forceinline__ void stage_tile_async(const float* __restrict__ src, int myrow,
                                                 float (*Xs)[kLda], int lane, uint64_t pol) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = i * 32 + lane;
    const int r = c >> 3, q = c & 7;
    const int rid = __shfl_sync(0xffffffffu, myrow, r);
    cp_async16_hint(&Xs[r][4 * q], src + (int64_t)(rid >= 0 ? rid : 0) * kH + 4 * q, rid >= 0 ? 16 : 0, pol);
  }
}

__device__ __forceinline__ void store_tile_rows(float* __restrict__ dst, int myrow,
                                                const float (*Ts)[kLda], int lane, uint64_t pol) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = i * 32 + lane;
    const int r = c >> 3, q = c & 7;
    const int rid = __shfl_sync(0xffffffffu, myrow, r);
    if (rid >= 0)
      st_f4_hint(dst + (int64_t)rid * kH + 4 * q, *reinterpret_cast<const float4*>(&Ts[r][4 * q]), pol);
  }
}

// Dense tail of a 16-row tile.  In: Hs = h rows, Xs = residual operand rows; lanes 0..15 hold the
// tile's row ids (myrow, -1 = no row) and per-source factors (mypre).
__device__ __forceinline__ void fwd_tile_tail(const LayerFwdArgs& a, float (*Xs)[kLda],
                                              float (*Hs)[kLda], const float* __restrict__ planes,
                                              int myrow, float mypre, int lane, uint64_t pol) {
  const int g = lane >> 2, t = lane & 3;
  float acc[kH / 8][4];
  float os[2] = {1.f, 1.f};
  if (a.out_scale) {
    const float mine = myrow >= 0 ? __ldg(a.out_scale + myrow) : 1.f;
    os[0] = __shfl_sync(0xffffffffu, mine, g);
    os[1] = __shfl_sync(0xffffffffu, mine, g + 8);
  }
  if (a.x) {
    warp_gemm16<kH, kH>(&Xs[0][0], kLda, planes, planes + kPlane, kLdb, acc, lane);
    __syncwarp();  // every lane's A fragments are read before the tile is overwritten
  }
#pragma unroll
  for (int j = 0; j < kH / 8; ++j) {
    const int c = 8 * j + 2 * t;
    float b0 = 0.f, b1 = 0.f;
    if (a.x && a.res_b) {
      b0 = __ldg(a.res_b + c);
      b1 = __ldg(a.res_b + c + 1);
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int rr = g + 8 * half;
      const float2 hv = *reinterpret_cast<const float2*>(&Hs[rr][c]);
      float v0, v1;
      if (a.x) {
        v0 = (acc[j][2 * half] + b0) + hv.x;
        v1 = (acc[j][2 * half + 1] + b1) + hv.y;
      } else {
        const float2 rv = *reinterpret_cast<const float2*>(&Xs[rr][c]);
        v0 = hv.x + rv.x;
        v1 = hv.y + rv.y;
      }
      if (a.act_out == 1) {
        v0 = v0 > 0.f ? v0 : 0.f;
        v1 = v1 > 0.f ? v1 : 0.f;
      }
      *reinterpret_cast<float2*>(&Xs[rr][c]) = make_float2(v0 * os[half], v1 * os[half]);
    }
  }
  __syncwarp();
  store_tile_rows(a.x_next, myrow, Xs, lane, pol);
  if (a.w_next) {
    warp_gemm16<kH, kH>(&Xs[0][0], kLda, planes + 2 * kPlane, planes + 3 * kPlane, kLdb, acc, lane);
    const float p0 = __shfl_sync(0xffffffffu, mypre, g);
    const float p1 = __shfl_sync(0xffffffffu, mypre, g + 8);
#pragma unroll
    for (int j = 0; j < kH / 8; ++j) {
      const int c = 8 * j + 2 * t;
      *reinterpret_cast<float2*>(&Hs[g][c]) = make_float2(acc[j][0] * p0, acc[j][1] * p0);
      *reinterpret_cast<float2*>(&Hs[g + 8][c]) = make_float2(acc[j][2] * p1, acc[j][3] * p1);
    }
    __syncwarp();
    store_tile_rows(a.m_next, myrow, Hs, lane, pol);
  }
  __syncwarp();  // tile buffers are free for the next tile
}

#ifndef MGCN_FWD_WARPS
#define MGCN_FWD_WARPS 4   // 4 warps x 5 CTAs/SM at 96 registers: 20 resident warps (0.84 ms vs 0.86 for 8 x 2)
#endif
constexpr int kFwdWarps = MGCN_FWD_WARPS;
constexpr int kFwdSmemFloats = 4 * kPlane + kFwdWarps * 2 * 16 * kLda;

__device__ __forceinline__ void fwd_fill_planes(const LayerFwdArgs& a, float* planes, int tid, int nthreads) {
  if (a.x) fill_plane(a.res_w, 1, kH, planes, planes + kPlane, tid, nthreads);                 // (k,c) = R[c][k]
  if (a.w_next) fill_plane(a.w_next, kH, 1, planes + 2 * kPlane, planes + 3 * kPlane, tid, nthreads);  // W[k][c]
}

__global__ void __launch_bounds__(kFwdWarps * 32, MGCN_FWD_MINB) k_layer_fwd(const LayerFwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* planes = smem;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float (*Xs)[kLda] = reinterpret_cast<float (*)[kLda]>(smem + 4 * kPlane + warp * 2 * 16 * kLda);
  float (*Hs)[kLda] = Xs + 16;
  fwd_fill_planes(a, planes, tid, kFwdWarps * 32);
  __syncthreads();

  const int sub = lane & 3, grp = lane >> 2, grp_lane0 = grp * 4;
  const unsigned gmask = 0xfu << grp_lane0;
  const int col = sub * 8;
  int64_t nseg = 0;
  if (a.seg_count) {
    nseg = *a.seg_count;
    if (nseg > a.seg_cap) nseg = a.seg_cap;
  }
  const int64_t limit = a.n_rows + nseg;          // tasks in work order: rows and hub segments mixed
  const int64_t n_tiles = (limit + 15) >> 4;
  const int64_t stride = (int64_t)gridDim.x * kFwdWarps;
  const uint64_t pol = policy_evict_first();

  int64_t tile = (int64_t)blockIdx.x * kFwdWarps + warp;
  if (a.tasks == nullptr) {
    // row-local mode (first layer, aggregated before the transform): a.m holds the finished
    // pre-activation z = post * (A_hat x) W of every row; tiles are 16 consecutive rows
    const int64_t n_loc = (a.n_rows + 15) >> 4;
    for (; tile < n_loc; tile += stride) {
      const int64_t r = tile * 16 + lane;
      const int myrow = (lane < 16 && r < a.n_rows) ? (int)r : -1;
      float mypre = 1.f;
      if (myrow >= 0 && a.pre && a.w_next) mypre = __ldg(a.pre + myrow);
      stage_tile_async(a.x ? a.x : a.resid, myrow, Xs, lane, pol);
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const int rowp = __shfl_sync(0xffffffffu, myrow, 8 * p + grp);
        if (rowp >= 0) {
          const Row8 z = ld_row8(a.m + (int64_t)rowp * kH + col);
          finish_h(a, z, 1.f, rowp, &Hs[8 * p + grp][0], sub, gmask, col);
        }
      }
      cp_async_wait_all();
      __syncwarp();
      fwd_tile_tail(a, Xs, Hs, planes, myrow, mypre, lane, pol);
    }
    return;
  }
  int4 dn = make_int4(-1, 0, 0, 0);
  if (tile < n_tiles) dn = load_tile_desc(a.tasks, tile * 16, limit, lane, pol);
  for (; tile < n_tiles; tile += stride) {
    const int4 d = dn;
    if (tile + stride < n_tiles) dn = load_tile_desc(a.tasks, (tile + stride) * 16, limit, lane, pol);
    const int myrow = (d.x >= 0 && d.w == 0) ? d.x : -1;   // rows this tile finishes (lanes 0..15)
    float mypost = 1.f, mypre = 1.f;
    if (myrow >= 0) {
      if (a.post) mypost = __ldg(a.post + myrow);
      if (a.pre && a.w_next) mypre = __ldg(a.pre + myrow);
    }
    // pass p: group g sums task 8p + g; first two index batches of both passes are fetched up front
    int beg[2], end[2], gi[2], gin[2];
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      beg[p] = __shfl_sync(0xffffffffu, d.y, 8 * p + grp);
      end[p] = __shfl_sync(0xffffffffu, d.z, 8 * p + grp);
      gi[p] = (beg[p] + sub < end[p]) ? ld_i32_hint(a.nbr_w + beg[p] + sub, pol) : 0;
      gin[p] = (beg[p] + 4 + sub < end[p]) ? ld_i32_hint(a.nbr_w + beg[p] + 4 + sub, pol) : 0;
    }
    stage_tile_async(a.x ? a.x : a.resid, myrow, Xs, lane, pol);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const int rowp = __shfl_sync(0xffffffffu, d.x, 8 * p + grp);
      const int slot = __shfl_sync(0xffffffffu, d.w, 8 * p + grp);
      const float postp = __shfl_sync(0xffffffffu, mypost, 8 * p + grp);
      if (rowp >= 0) {
        const Row8 acc = gather_sum(a.m, a.nbr_w, beg[p], end[p], gi[p], gin[p], sub, grp_lane0, gmask, col, pol);
        if (slot != 0) {
          store_partial(a.partial, slot, col, acc);
        } else {
          finish_h(a, acc, postp, rowp, &Hs[8 * p + grp][0], sub, gmask, col);
        }
      }
    }
    cp_async_wait_all();
    __syncwarp();
    fwd_tile_tail(a, Xs, Hs, planes, myrow, mypre, lane, pol);
  }
}

// First layer with a narrow input (mgcn_gcn_first_layer_fwd): row-local, z and the residual term are formed in
// the kernel from the [N, nhin] operands; then the same tile tail.
__global__ void __launch_bounds__(kFwdWarps * 32, 4) k_first_layer_fwd(const LayerFwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* planes = smem;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float (*Xs)[kLda] = reinterpret_cast<float (*)[kLda]>(smem + 4 * kPlane + warp * 2 * 16 * kLda);
  float (*Hs)[kLda] = Xs + 16;
  fwd_fill_planes(a, planes, tid, kFwdWarps * 32);
  float* nws = planes;   // W_in [k][c] at 0, R^T [k][c] at 128, r at 256 (the residual planes are unused: a.x == NULL)
  for (int i = tid; i < a.nhin * kH; i += kFwdWarps * 32) {
    const int k = i / kH, c = i % kH;
    nws[i] = __ldg(a.nw + i);
    nws[128 + i] = __ldg(a.res_w + c * a.nhin + k);
  }
  if (tid < kH) nws[256 + tid] = a.res_b ? __ldg(a.res_b + tid) : 0.f;
  __syncthreads();
  const int sub = lane & 3, grp = lane >> 2;
  const unsigned gmask = 0xfu << (grp * 4);
  const int col = sub * 8;
  const uint64_t pol = policy_evict_first();
  const int64_t n_loc = (a.n_rows + 15) >> 4;
  for (int64_t tile = (int64_t)blockIdx.x * kFwdWarps + warp; tile < n_loc; tile += (int64_t)gridDim.x * kFwdWarps) {
    const int64_t r = tile * 16 + lane;
    const int myrow = (lane < 16 && r < a.n_rows) ? (int)r : -1;
    float mypre = 1.f;
    if (myrow >= 0 && a.pre && a.w_next) mypre = __ldg(a.pre + myrow);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const int rowp = __shfl_sync(0xffffffffu, myrow, 8 * p + grp);
      if (rowp >= 0) {
        Row8 z, rs;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          z.v[q] = 0.f;
          rs.v[q] = 0.f;
        }
        for (int k = 0; k < a.nhin; ++k) {
          const float sv = __ldg(a.ns + (int64_t)rowp * a.nhin + k);
          const float xv = __ldg(a.nx + (int64_t)rowp * a.nhin + k);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            z.v[q] = fmaf(sv, nws[k * kH + col + q], z.v[q]);
            rs.v[q] = fmaf(xv, nws[128 + k * kH + col + q], rs.v[q]);
          }
        }
        const float ps = a.npost ? __ldg(a.npost + rowp) : 1.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          z.v[q] *= ps;
          rs.v[q] += nws[256 + col + q];
        }
        float* xr = &Xs[8 * p + grp][col];
        *reinterpret_cast<float4*>(xr) = make_float4(rs.v[0], rs.v[1], rs.v[2], rs.v[3]);
        *reinterpret_cast<float4*>(xr + 4) = make_float4(rs.v[4], rs.v[5], rs.v[6], rs.v[7]);
        finish_h(a, z, 1.f, rowp, &Hs[8 * p + grp][0], sub, gmask, col);
      }
    }
    __syncwarp();
    fwd_tile_tail(a, Xs, Hs, planes, myrow, mypre, lane, pol);
  }
}

// The same layer without a following transform (w_next == NULL: the aggregate-then-transform stack): nothing needs a
// tile — a lane group of 4 owns a row, 8 columns per lane, the operations and their order are those of
// k_first_layer_fwd + fwd_tile_tail (identical results), the outputs leave as whole 128-byte rows.  A pure streaming pass.
__global__ void __launch_bounds__(256) k_first_layer_fwd_stream(const LayerFwdArgs a) {
  __shared__ float nws[288];   // W_in [k][c] at 0, R^T [k][c] at 128, r at 256
  const int tid = threadIdx.x, lane = tid & 31;
  for (int i = tid; i < a.nhin * kH; i += 256) {
    const int k = i / kH, c = i % kH;
    nws[i] = __ldg(a.nw + i);
    nws[128 + i] = __ldg(a.res_w + c * a.nhin + k);
  }
  if (tid < kH) nws[256 + tid] = a.res_b ? __ldg(a.res_b + tid) : 0.f;
  __syncthreads();
  const int sub = lane & 3, col = sub * 8;
  const unsigned gmask = 0xfu << (lane & ~3);
  const uint64_t pol = policy_evict_first();
  const int64_t groups = (int64_t)gridDim.x * 64;
  for (int64_t row = (int64_t)blockIdx.x * 64 + (tid >> 2); row < a.n_rows; row += groups) {
    Row8 z, rs;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      z.v[q] = 0.f;
      rs.v[q] = 0.f;
    }
    for (int k = 0; k < a.nhin; ++k) {
      const float sv = __ldg(a.ns + row * a.nhin + k);
      const float xv = __ldg(a.nx + row * a.nhin + k);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        z.v[q] = fmaf(sv, nws[k * kH + col + q], z.v[q]);
        rs.v[q] = fmaf(xv, nws[128 + k * kH + col + q], rs.v[q]);
      }
    }
    const float ps = a.npost ? __ldg(a.npost + row) : 1.f;
    const float os = a.out_scale ? __ldg(a.out_scale + row) : 1.f;
    const uint32_t kept = a.keep ? __ldg(a.keep + row) >> col : 0xffu;
    uint32_t bits = 0;
    float o[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float h = z.v[q] * ps;
      if (a.bias) h = __fadd_rn(h, __ldg(a.bias + col + q));
      h = h > 0.f ? h : 0.f;
      if (a.keep) h = ((kept >> q) & 1u) ? __fmul_rn(h, a.keep_scale) : 0.f;   // dropout (see gcn_fwd_tc.cu)
      bits |= (h > 0.f ? 1u : 0u) << q;
      float v = h + (rs.v[q] + nws[256 + col + q]);
      if (a.act_out == 1) v = v > 0.f ? v : 0.f;
      o[q] = v * os;
    }
    bits <<= col;
    bits |= __shfl_xor_sync(gmask, bits, 1);
    bits |= __shfl_xor_sync(gmask, bits, 2);
    if (sub == 0) a.hmask[row] = bits;
    float* out = a.x_next + row * kH + col;
    st_f4_hint(out, make_float4(o[0], o[1], o[2], o[3]), pol);
    st_f4_hint(out + 4, make_float4(o[4], o[5], o[6], o[7]), pol);
  }
}

// hub rows: partial sums of the row's segments added left to right, then the same tile tail
__global__ void __launch_bounds__(kFwdWarps * 32, 2) k_layer_fwd_hubs(const LayerFwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* planes = smem;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float (*Xs)[kLda] = reinterpret_cast<float (*)[kLda]>(smem + 4 * kPlane + warp * 2 * 16 * kLda);
  float (*Hs)[kLda] = Xs + 16;
  int64_t nh = *a.hub_count;
  if (nh > a.hub_cap) nh = a.hub_cap;
  const int64_t n_tiles = (nh + 15) >> 4;
  if ((int64_t)blockIdx.x * kFwdWarps >= n_tiles) return;
  fwd_fill_planes(a, planes, tid, kFwdWarps * 32);
  __syncthreads();
  const int sub = lane & 3, grp = lane >> 2, grp_lane0 = grp * 4;
  const unsigned gmask = 0xfu << grp_lane0;
  const int col = sub * 8;
  const uint64_t pol = policy_evict_first();
  for (int64_t tile = (int64_t)blockIdx.x * kFwdWarps + warp; tile < n_tiles;
       tile += (int64_t)gridDim.x * kFwdWarps) {
    int myrow = -1, myseg0 = 0, mynseg = 0;
    float mypost = 1.f, mypre = 1.f;
    const int64_t k = tile * 16 + lane;
    if (lane < 16 && k < nh) {
      myrow = __ldg(a.hub_rows + k);
      myseg0 = __ldg(a.hub_seg0 + k);
      const int len = __ldg(a.rowptr + myrow + 1) - __ldg(a.rowptr + myrow);
      mynseg = (len + a.hub_threshold - 1) / a.hub_threshold;
      if (a.post) mypost = __ldg(a.post + myrow);
      if (a.pre && a.w_next) mypre = __ldg(a.pre + myrow);
    }
    stage_tile_async(a.x ? a.x : a.resid, myrow, Xs, lane, pol);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const int rowp = __shfl_sync(0xffffffffu, myrow, 8 * p + grp);
      const int s0 = __shfl_sync(0xffffffffu, myseg0, 8 * p + grp);
      const int ns = __shfl_sync(0xffffffffu, mynseg, 8 * p + grp);
      const float postp = __shfl_sync(0xffffffffu, mypost, 8 * p + grp);
      if (rowp >= 0) {
        Row8 tot = sum_partials(a.partial, s0, 1, col);   // reduced by k_hub_reduce
        finish_h(a, tot, postp, rowp, &Hs[8 * p + grp][0], sub, gmask, col);
      }
    }
    cp_async_wait_all();
    __syncwarp();
    fwd_tile_tail(a, Xs, Hs, planes, myrow, mypre, lane, pol);
  }
}

// -------------------------------------------------------------------------------------------------
// plain aggregation on the same flat gather (the transposed pass of the backward):
//   out_i = act( post_i * sum_k x[nbr_k] )
// -------------------------------------------------------------------------------------------------
struct AggFlatArgs {
  const int4* tasks;
  const int32_t* nbr_w;
  const int32_t* seg_count;
  const int32_t* hub_rows;
  const int32_t* hub_seg0;
  const int32_t* hub_count;
  const int32_t* rowptr;
  const float* x;
  const float* post;
  float* out;
  float* partial;
  int64_t n_rows;
  int64_t seg_cap;
  int64_t hub_cap;
  int act;
  int hub_threshold;
};

__device__ __forceinline__ void agg_finish_row(const AggFlatArgs& a, Row8 acc, float ps, int64_t row,
                                               int col, uint64_t pol) {
  if (a.post) {
#pragma unroll
    for (int q = 0; q < 8; ++q) acc.v[q] = __fmul_rn(acc.v[q], ps);
  }
  if (a.act == 1) {
#pragma unroll
    for (int q = 0; q < 8; ++q) acc.v[q] = acc.v[q] > 0.f ? acc.v[q] : 0.f;
  }
  float* o = a.out + row * kH + col;
  st_f4_hint(o, make_float4(acc.v[0], acc.v[1], acc.v[2], acc.v[3]), pol);
  st_f4_hint(o + 4, make_float4(acc.v[4], acc.v[5], acc.v[6], acc.v[7]), pol);
}

__global__ void __launch_bounds__(MGCN_AGG_WARPS * 32, MGCN_AGG_MINB) k_agg_flat(const AggFlatArgs a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  const int sub = lane & 3, grp = lane >> 2, grp_lane0 = grp * 4;
  const unsigned gmask = 0xfu << grp_lane0;
  const int col = sub * 8;
  int64_t nseg = 0;
  if (a.seg_count) {
    nseg = *a.seg_count;
    if (nseg > a.seg_cap) nseg = a.seg_cap;
  }
  const int64_t limit = a.n_rows + nseg;
  const int64_t n_tiles = (limit + 15) >> 4;
  const int64_t stride = (int64_t)gridDim.x * MGCN_AGG_WARPS;
  const uint64_t pol = policy_evict_first();
  int64_t tile = (int64_t)blockIdx.x * MGCN_AGG_WARPS + warp;
  int4 dn = make_int4(-1, 0, 0, 0);
  if (tile < n_tiles) dn = load_tile_desc(a.tasks, tile * 16, limit, lane, pol);
  for (; tile < n_tiles; tile += stride) {
    const int4 d = dn;
    if (tile + stride < n_tiles) dn = load_tile_desc(a.tasks, (tile + stride) * 16, limit, lane, pol);
    float mypost = 1.f;
    if (a.post && d.x >= 0 && d.w == 0) mypost = __ldg(a.post + d.x);
    int beg[2], end[2], gi[2], gin[2];
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      beg[p] = __shfl_sync(0xffffffffu, d.y, 8 * p + grp);
      end[p] = __shfl_sync(0xffffffffu, d.z, 8 * p + grp);
      gi[p] = (beg[p] + sub < end[p]) ? ld_i32_hint(a.nbr_w + beg[p] + sub, pol) : 0;
      gin[p] = (beg[p] + 4 + sub < end[p]) ? ld_i32_hint(a.nbr_w + beg[p] + 4 + sub, pol) : 0;
    }
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const int rowp = __shfl_sync(0xffffffffu, d.x, 8 * p + grp);
      const int slot = __shfl_sync(0xffffffffu, d.w, 8 * p + grp);
      const float postp = __shfl_sync(0xffffffffu, mypost, 8 * p + grp);
      if (rowp >= 0) {
        const Row8 acc = gather_sum(a.x, a.nbr_w, beg[p], end[p], gi[p], gin[p], sub, grp_lane0, gmask, col, pol);
        if (slot != 0) {
          store_partial(a.partial, slot, col, acc);
        } else {
          agg_finish_row(a, acc, postp, rowp, col, pol);
        }
      }
    }
  }
}

// k_hub_reduce and the finishing pass over the hub rows in one launch: the warp (or, for giant hubs, the CTA) that has summed a hub row's
// segment partials — same runs, same order, same sums — finishes the row itself instead of storing the sum for a
// second kernel.  One launch less per aggregation (11 per botnet step).
__global__ void __launch_bounds__(256) k_agg_flat_hub_finish(const AggFlatArgs a) {
  __shared__ int giant_k[kGiantList];
  __shared__ int n_giant;
  __shared__ __align__(16) float red[64][kH];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane & 3, grp = lane >> 2, col = sub * 8;
  int64_t nh = *a.hub_count;
  if (nh > a.hub_cap) nh = a.hub_cap;
  const uint64_t pol = policy_evict_first();
  const int64_t W = (int64_t)gridDim.x * 8;
  int64_t k = (int64_t)blockIdx.x * 8 + warp;
  // rounds, as in k_hub_reduce: every giant gets the 64-run grouping whatever the grid and the hub table order
  bool more = true;
  while (more) {
    if (threadIdx.x == 0) n_giant = 0;
    __syncthreads();
    for (; k < nh; k += W) {
      const int64_t row = __ldg(a.hub_rows + k);
      const int s0 = __ldg(a.hub_seg0 + k);
      const int len = __ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row);
      const int ns = (len + a.hub_threshold - 1) / a.hub_threshold;
      if (ns > kGiantSegs) {   // queue for the CTA-wide pass below (the slot order never reaches the results)
        int slot = 0;
        if (lane == 0) slot = atomicAdd(&n_giant, 1);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot >= kGiantList) break;   // list full: this hub waits for the next round
        if (lane == 0) giant_k[slot] = (int)k;
        continue;
      }
      Row8 tot;
      if (ns <= 1) {
        tot = sum_partials(a.partial, s0, 1, col);
      } else {
        const int per = (ns + 7) >> 3;
        const Row8 run = hub_run_sum(a.partial, s0, grp * per, min(ns, grp * per + per), col);
        tot = run;   // group 0: its own run; then runs 1..7 in order
#pragma unroll
        for (int g = 1; g < 8; ++g) {
          Row8 other;
#pragma unroll
          for (int q = 0; q < 8; ++q) other.v[q] = __shfl_sync(0xffffffffu, run.v[q], 4 * g + sub);
          if (g * per < ns) row8_add(tot, other);
        }
      }
      if (grp == 0) agg_finish_row(a, tot, a.post ? __ldg(a.post + row) : 1.f, row, col, pol);
    }
    __syncthreads();
    // giants: 64 lane groups of the CTA sum 64 contiguous runs concurrently, group 0 adds the 64 run sums in order
    const int ng = min(n_giant, kGiantList);
    for (int gi = 0; gi < ng; ++gi) {
      const int64_t k = giant_k[gi];
      const int64_t row = __ldg(a.hub_rows + k);
      const int s0 = __ldg(a.hub_seg0 + k);
      const int len = __ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row);
      const int ns = (len + a.hub_threshold - 1) / a.hub_threshold;
      const int per = (ns + 63) >> 6, gid = warp * 8 + grp;
      const Row8 run = hub_run_sum(a.partial, s0, gid * per, min(ns, gid * per + per), col);
      *reinterpret_cast<float4*>(&red[gid][col]) = make_float4(run.v[0], run.v[1], run.v[2], run.v[3]);
      *reinterpret_cast<float4*>(&red[gid][col + 4]) = make_float4(run.v[4], run.v[5], run.v[6], run.v[7]);
      __syncthreads();
      if (warp == 0 && grp == 0) {
        Row8 tot = run;
        for (int g = 1; g < 64 && g * per < ns; ++g) {
          const float4 lo = *reinterpret_cast<const float4*>(&red[g][col]), hi = *reinterpret_cast<const float4*>(&red[g][col + 4]);
          Row8 o;
          o.v[0] = lo.x; o.v[1] = lo.y; o.v[2] = lo.z; o.v[3] = lo.w;
          o.v[4] = hi.x; o.v[5] = hi.y; o.v[6] = hi.z; o.v[7] = hi.w;
          row8_add(tot, o);
        }
        agg_finish_row(a, tot, a.post ? __ldg(a.post + row) : 1.f, row, col, pol);
      }
      __syncthreads();
    }
    more = __syncthreads_or(k < nh) != 0;
  }
}

// called by mgcn_aggregate_prescaled (agg_pipelined.cu) for H = 32 without bias / residual / mean
int launch_agg_flat32(const mgcn_csr_t* g, const float* x, const float* post, int act, float* out,
                      float* partial, bool hubs, void* stream) {
  AggFlatArgs a{};
  a.tasks = reinterpret_cast<const int4*>(g->tasks);
  a.nbr_w = g->nbr_w;
  a.seg_count = hubs ? g->seg_count : nullptr;
  a.hub_rows = g->hub_rows;
  a.hub_seg0 = g->hub_seg0;
  a.hub_count = g->hub_count;
  a.rowptr = g->rowptr;
  a.x = x;
  a.post = post;
  a.out = out;
  a.partial = partial;
  a.n_rows = g->n_rows;
  a.seg_cap = hubs ? g->seg_cap : 0;
  a.hub_cap = hubs ? g->hub_cap : 0;
  a.act = act;
  a.hub_threshold = g->hub_threshold;
  const int64_t max_tiles = ceil_div(g->n_rows + a.seg_cap, 16);
  int64_t blocks = ceil_div(max_tiles, MGCN_AGG_WARPS);
  if (blocks > (int64_t)kNumSMs * MGCN_AGG_MINB) blocks = (int64_t)kNumSMs * MGCN_AGG_MINB;
  MGCN_LAUNCH(k_agg_flat, (unsigned)blocks, MGCN_AGG_WARPS * 32, 0, stream, a);
  if (hubs) {
    int64_t hb = ceil_div(a.hub_cap, 8);
    if (hb > (int64_t)kNumSMs * 8) hb = (int64_t)kNumSMs * 8;
    MGCN_LAUNCH(k_agg_flat_hub_finish, (unsigned)hb, 256, 0, stream, a);
  }
  return MGCN_OK;
}

// -------------------------------------------------------------------------------------------------
// backward, row-local
// -------------------------------------------------------------------------------------------------
struct LayerBwdArgs {
  const float* dxw;          // [N,32]  pre * A^T gs          (transposed aggregation)
  const float* gy;           // [N,32]  gradient w.r.t. y_n
  const float* x;            // [N,32]  layer input x_n
  const float* w;            // weight_node (in, out)
  const float* res_w;        // residual weight (out, in)
  const uint32_t* hmask_prev;  // bits of h_{n-1} > 0
  const float* post;         // per-target factor or NULL
  float* gy_prev;            // [N,32] or NULL
  float* gs_prev;            // [N,32] or NULL
  float* part_w;             // [grid][32*32]
  float* part_r;             // [grid][32*32]
  float* part_b;             // [grid][32]
  int64_t n_rows;
};

constexpr int kBwdWarps = 8;
constexpr int kBwdRows = 16 * kBwdWarps;  // rows per CTA tile
constexpr int kLdx = kH + 8;              // x tile: only ever a transposed-product operand
constexpr int kBwdSmemFloats = 4 * kPlane + kBwdRows * (2 * kLda + kLdx);

template <int LD>
__device__ __forceinline__ void stage_rows_async(const float* __restrict__ src, int64_t row0, int64_t N,
                                                 float (*dst)[LD], int tid, uint64_t pol) {
#pragma unroll
  for (int i = 0; i < kBwdRows * 8 / (kBwdWarps * 32); ++i) {
    const int c = i * (kBwdWarps * 32) + tid;
    const int r = c >> 3, q = c & 7;
    const int64_t gr = row0 + r;
    cp_async16_hint(&dst[r][4 * q], src + (gr < N ? gr : 0) * kH + 4 * q, gr < N ? 16 : 0, pol);
  }
}

// 16 rows of a tile -> global, 128 bytes per row, 4 rows per instruction
__device__ __forceinline__ void store_rows16(float* __restrict__ dst, int64_t row0, int64_t N,
                                             const float (*src)[kLda], int lane, uint64_t pol) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = i * 32 + lane;
    const int r = c >> 3, q = c & 7;
    const int64_t gr = row0 + r;
    if (gr < N) st_f4_hint(dst + gr * kH + 4 * q, *reinterpret_cast<const float4*>(&src[r][4 * q]), pol);
  }
}

// One CTA walks 128-row tiles.  Row-local products (G): warp w owns rows [16w, 16w+16).  Weight
// gradients: warp w owns one 16x16 block of dW (w < 4) or dR (w >= 4) over all 128 rows of the tile,
// so the persistent accumulators are 8 registers per thread and no cross-warp reduction is needed.
__global__ void __launch_bounds__(kBwdWarps * 32, 2) k_layer_bwd(const LayerBwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* planes = smem;  // W^T hi/lo, R hi/lo
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  float (*Dw)[kLda] = reinterpret_cast<float (*)[kLda]>(smem + 4 * kPlane);
  float (*Gy)[kLda] = Dw + kBwdRows;
  float (*Xs)[kLdx] = reinterpret_cast<float (*)[kLdx]>(smem + 4 * kPlane + 2 * kBwdRows * kLda);
  fill_plane(a.w, 1, kH, planes, planes + kPlane, tid, kBwdWarps * 32);                  // (k=c, n=j) = W[j][c]
  fill_plane(a.res_w, kH, 1, planes + 2 * kPlane, planes + 3 * kPlane, tid, kBwdWarps * 32);  // (k=c, n=j) = R[c][j]
  const int prod = warp >> 2;            // 0: dW = x^T dxw, 1: dR = gy^T x
  const int m0 = ((warp >> 1) & 1) * 16, n0 = (warp & 1) * 16;
  float acc_blk[2][4];
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc_blk[j][q] = 0.f;
  float acc_b = 0.f;
  const bool want_prev = a.gy_prev != nullptr;
  const uint64_t pol = policy_evict_first();
  const int64_t ntiles = (a.n_rows + kBwdRows - 1) / kBwdRows;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * kBwdRows;
    __syncthreads();  // previous tile fully consumed (also orders the plane fill)
    stage_rows_async<kLda>(a.dxw, row0, a.n_rows, Dw, tid, pol);
    stage_rows_async<kLda>(a.gy, row0, a.n_rows, Gy, tid, pol);
    stage_rows_async<kLdx>(a.x, row0, a.n_rows, Xs, tid, pol);
    uint32_t mybits = 0;
    float mypost = 1.f;
    const int64_t myrow = row0 + warp * 16 + lane;
    if (want_prev && lane < 16 && myrow < a.n_rows) {
      mybits = __ldg(a.hmask_prev + myrow);
      if (a.post) mypost = __ldg(a.post + myrow);
    }
    cp_async_wait_all();
    __syncthreads();
    // weight-gradient block of this warp over the 128 rows, flushed to the RN accumulators every 32
    {
      const float* As = prod == 0 ? &Xs[0][0] : &Gy[0][0];
      const int lda = prod == 0 ? kLdx : kLda;
      const float* Bs = prod == 0 ? &Dw[0][0] : &Xs[0][0];
      const int ldb = prod == 0 ? kLda : kLdx;
#pragma unroll 1
      for (int rc = 0; rc < kBwdRows; rc += 32) {
        float mainc[2][4], corr[2][4];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int q = 0; q < 4; ++q) mainc[j][q] = corr[j][q] = 0.f;
#pragma unroll
        for (int r0 = rc; r0 < rc + 32; r0 += 8) {
          uint32_t ahi[4], alo[4];
          split_tf32(As[(r0 + t) * lda + m0 + g], ahi[0], alo[0]);
          split_tf32(As[(r0 + t) * lda + m0 + g + 8], ahi[1], alo[1]);
          split_tf32(As[(r0 + t + 4) * lda + m0 + g], ahi[2], alo[2]);
          split_tf32(As[(r0 + t + 4) * lda + m0 + g + 8], ahi[3], alo[3]);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint32_t bhi[2], blo[2];
            split_tf32(Bs[(r0 + t) * ldb + n0 + 8 * j + g], bhi[0], blo[0]);
            split_tf32(Bs[(r0 + t + 4) * ldb + n0 + 8 * j + g], bhi[1], blo[1]);
            mma_tf32_16x8x8(corr[j], alo, bhi);
            mma_tf32_16x8x8(corr[j], ahi, blo);
            mma_tf32_16x8x8(mainc[j], ahi, bhi);
          }
        }
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc_blk[j][q] += mainc[j][q] + corr[j][q];
      }
      float colsum = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) colsum += Gy[warp * 16 + r][lane];
      acc_b += colsum;
    }
    if (want_prev) {
      __syncthreads();  // every warp is done reading all rows of Dw / Gy
      float (*Dt)[kLda] = Dw + warp * 16;
      float (*Gt)[kLda] = Gy + warp * 16;
      float accg[4][4], second[4][4];
      warp_gemm16<kH, kH>(&Dt[0][0], kLda, planes, planes + kPlane, kLdb, accg, lane);
      warp_gemm16<kH, kH>(&Gt[0][0], kLda, planes + 2 * kPlane, planes + 3 * kPlane, kLdb, second, lane);
      __syncwarp();  // all fragment reads of this warp's rows are done
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int rr = g + 8 * half;
        const uint32_t bits = __shfl_sync(0xffffffffu, mybits, rr);
        const float ps = __shfl_sync(0xffffffffu, mypost, rr);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = 8 * j + 2 * t;
          const float2 xv = *reinterpret_cast<const float2*>(&Xs[warp * 16 + rr][c]);
          const float g0 = xv.x > 0.f ? accg[j][2 * half] + second[j][2 * half] : 0.f;
          const float g1 = xv.y > 0.f ? accg[j][2 * half + 1] + second[j][2 * half + 1] : 0.f;
          *reinterpret_cast<float2*>(&Dt[rr][c]) = make_float2(g0, g1);
          const float s0 = ((bits >> c) & 1u) ? g0 * ps : 0.f;
          const float s1 = ((bits >> (c + 1)) & 1u) ? g1 * ps : 0.f;
          *reinterpret_cast<float2*>(&Gt[rr][c]) = make_float2(s0, s1);
        }
      }
      __syncwarp();
      store_rows16(a.gy_prev, row0 + warp * 16, a.n_rows, Dt, lane, pol);
      store_rows16(a.gs_prev, row0 + warp * 16, a.n_rows, Gt, lane, pol);
    }
  }
  // this warp's 16x16 block of dW (row = input j, col = output c) or dR (row = output c, col = input j)
  float* part = (prod == 0 ? a.part_w : a.part_r) + (int64_t)blockIdx.x * kH * kH;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int c = n0 + 8 * j + 2 * t;
    *reinterpret_cast<float2*>(part + (m0 + g) * kH + c) = make_float2(acc_blk[j][0], acc_blk[j][1]);
    *reinterpret_cast<float2*>(part + (m0 + g + 8) * kH + c) = make_float2(acc_blk[j][2], acc_blk[j][3]);
  }
  __syncthreads();
  float* red = smem + 4 * kPlane;
  red[warp * 32 + lane] = acc_b;
  __syncthreads();
  if (tid < 32) {
    float s = red[tid];
#pragma unroll
    for (int w = 1; w < kBwdWarps; ++w) s += red[w * 32 + tid];
    a.part_b[(int64_t)blockIdx.x * kH + tid] = s;
  }
}

// gs = post * gy * bits   (seed of the backward: last layer has no outer ReLU)
__global__ void __launch_bounds__(256) k_mask_bits_scale(const float* __restrict__ gy,
                                                         const uint32_t* __restrict__ bits,
                                                         const float* __restrict__ post, int64_t N,
                                                         float* __restrict__ gs) {
  const int64_t total = N * (kH / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i >> 3;
    const int c = (int)(i & 7) * 4;
    const uint32_t b = __ldg(bits + row) >> c;
    const float s = post ? __ldg(post + row) : 1.f;
    float4 v = __ldg(reinterpret_cast<const float4*>(gy) + i);
    v.x = (b & 1u) ? v.x * s : 0.f;
    v.y = (b & 2u) ? v.y * s : 0.f;
    v.z = (b & 4u) ? v.z * s : 0.f;
    v.w = (b & 8u) ? v.w * s : 0.f;
    reinterpret_cast<float4*>(gs)[i] = v;
  }
}

static int bwd_grid(int64_t N) {
  const int64_t tiles = ceil_div(N > 0 ? N : 1, kBwdRows);
  const int64_t p = (int64_t)kNumSMs * 2;
  return (int)(tiles < p ? tiles : p);
}

}  // namespace mgcn

using namespace mgcn;

extern "C" int mgcn_gcn_layer_fwd(const mgcn_csr_t* g, const float* m, int64_t n_in, const float* x,
                                  const float* resid, const float* res_w, const float* res_b,
                                  const float* w_next, const float* bias, const float* pre,
                                  const float* post, int act_out, int64_t H, float* x_next,
                                  float* m_next, uint32_t* hmask, void* workspace,
                                  size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H == kH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(act_out == 0 || act_out == 1, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(n_in >= 0 && (!g || g->n_rows >= 0), MGCN_ERR_RANGE);
  const bool local = g == nullptr;   // row-local mode: m is the finished pre-activation of row i
  const int64_t n_rows = local ? n_in : g->n_rows;
  const bool hubs = !local && g->hub_rows && g->hub_seg0 && g->hub_count && g->seg_count &&
                    g->hub_cap > 0 && g->seg_cap > 0;
  WorkspaceCarver ws(workspace);
  float* partial = ws.take<float>(hubs ? (size_t)g->seg_cap * kH : 0);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  if (n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(x_next && hmask && m, MGCN_ERR_NULL);
  MGCN_REQUIRE(local || (g->rowptr && g->tasks), MGCN_ERR_NULL);
  MGCN_REQUIRE((x != nullptr) != (resid != nullptr), MGCN_ERR_NULL);   // exactly one residual form
  MGCN_REQUIRE(!x || res_w, MGCN_ERR_NULL);
  MGCN_REQUIRE(!w_next || m_next, MGCN_ERR_NULL);
  MGCN_REQUIRE(local || g->nnz_cap == 0 || g->nbr_w, MGCN_ERR_NULL);
  MGCN_REQUIRE((reinterpret_cast<uintptr_t>(m) & 31u) == 0, MGCN_ERR_ALIGN);   // 256-bit row gathers
  MGCN_REQUIRE((local || aligned16(g->tasks)) && aligned16(x_next) && aligned16(partial) &&
                   (!x || aligned16(x)) && (!resid || aligned16(resid)) &&
                   (!m_next || aligned16(m_next)) && (!bias || aligned16(bias)),
               MGCN_ERR_ALIGN);
  LayerFwdArgs a{};
  if (!local) {
    a.tasks = reinterpret_cast<const int4*>(g->tasks);
    a.nbr_w = g->nbr_w;
    a.seg_count = hubs ? g->seg_count : nullptr;
    a.hub_rows = g->hub_rows;
    a.hub_seg0 = g->hub_seg0;
    a.hub_count = g->hub_count;
    a.rowptr = g->rowptr;
    a.hub_threshold = g->hub_threshold;
  }
  a.m = m; a.x = x; a.resid = resid; a.res_w = res_w; a.res_b = res_b; a.w_next = w_next;
  a.bias = bias; a.pre = pre; a.post = post;
  a.x_next = x_next; a.m_next = m_next; a.hmask = hmask; a.partial = partial;
  a.n_rows = n_rows;
  a.seg_cap = hubs ? g->seg_cap : 0;
  a.hub_cap = hubs ? g->hub_cap : 0;
  a.act_out = act_out;
  const size_t smem = sizeof(float) * kFwdSmemFloats;
  // the attribute belongs to (function, device): set on every call (cheap), so a second GPU in the same process
  // gets it too and a failure is reported every time
  cudaError_t attr_err = cudaSuccess;
  {
    attr_err = cudaFuncSetAttribute(k_layer_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(k_layer_fwd_hubs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  MGCN_CHECK_CUDA(attr_err);
  const int64_t max_tiles = ceil_div(n_rows + a.seg_cap, 16);
  int64_t blocks = ceil_div(max_tiles, kFwdWarps);
  if (blocks > (int64_t)kNumSMs * MGCN_FWD_MINB) blocks = (int64_t)kNumSMs * MGCN_FWD_MINB;
  MGCN_LAUNCH(k_layer_fwd, (unsigned)blocks, kFwdWarps * 32, smem, stream, a);
  if (hubs) {
    const int rc = launch_hub_reduce(g, partial, stream);
    if (rc != MGCN_OK) return rc;
    int64_t hb = ceil_div(ceil_div(a.hub_cap, 16), kFwdWarps);
    if (hb > (int64_t)kNumSMs * 4) hb = (int64_t)kNumSMs * 4;   // one 16-row tile per warp at the botnet batch
    MGCN_LAUNCH(k_layer_fwd_hubs, (unsigned)hb, kFwdWarps * 32, smem, stream, a);
  }
  return MGCN_OK;
}

// First layer of a stack whose input is narrow (H_in <= 4; the botnet model has H_in = 1): the layer is
// aggregated BEFORE its transform, s = sum_j pre_j x_j (mgcn_spmm on [N, H_in]), and this launch forms
//   h = relu( post * (s W_in) ),  y = h + x R^T + r,  x' = act(y),  m' = pre * (x' W_next)
// reading only the two [N, H_in] operands (gcn_base_models.py:201-240 + gcn_model.py:96-105 for layer 0).
extern "C" int mgcn_gcn_first_layer_fwd(const float* s, const float* x, int64_t N, int64_t Hin, const float* w_in,
                                        const float* res_w, const float* res_b, const float* w_next,
                                        const float* pre, const float* post, const float* out_scale, int act_out,
                                        int64_t H, float* x_next, float* m_next, uint32_t* hmask, void* stream) {
  return mgcn_gcn_first_layer_fwd_ex(s, x, N, Hin, w_in, res_w, res_b, w_next, pre, post, out_scale, nullptr, 1.f,
                                     act_out, H, x_next, m_next, hmask, stream);
}

extern "C" int mgcn_gcn_first_layer_fwd_ex(const float* s, const float* x, int64_t N, int64_t Hin, const float* w_in,
                                           const float* res_w, const float* res_b, const float* w_next,
                                           const float* pre, const float* post, const float* out_scale,
                                           const uint32_t* keep, float keep_scale, int act_out, int64_t H,
                                           float* x_next, float* m_next, uint32_t* hmask, void* stream) {
  return mgcn_gcn_first_layer_fwd_bias(s, x, N, Hin, w_in, res_w, res_b, nullptr, w_next, pre, post, out_scale, keep,
                                       keep_scale, act_out, H, x_next, m_next, hmask, stream);
}

// The same with the node-model bias b [32] (NodeModelAdditive's default bias=True), added where the reference adds it:
// h = relu(post * (s W_in) + b), before the dropout (both kernels: finish_h / the streaming epilogue).
extern "C" int mgcn_gcn_first_layer_fwd_bias(const float* s, const float* x, int64_t N, int64_t Hin, const float* w_in,
                                             const float* res_w, const float* res_b, const float* bias,
                                             const float* w_next, const float* pre, const float* post,
                                             const float* out_scale, const uint32_t* keep, float keep_scale,
                                             int act_out, int64_t H, float* x_next, float* m_next, uint32_t* hmask,
                                             void* stream) {
  MGCN_REQUIRE(H == kH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(!(keep && w_next), MGCN_ERR_SHAPE);   // dropout only in the streaming pass
  MGCN_REQUIRE(Hin >= 1 && Hin <= 4, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(act_out == 0 || act_out == 1, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N >= 0 && N < (int64_t(1) << 31), MGCN_ERR_RANGE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(s && x && w_in && res_w && x_next && hmask, MGCN_ERR_NULL);
  MGCN_REQUIRE(!w_next || m_next, MGCN_ERR_NULL);
  MGCN_REQUIRE(!(w_next && out_scale), MGCN_ERR_SHAPE);   // scaled rows would feed the next layer's messages
  MGCN_REQUIRE(aligned16(x_next) && (!m_next || aligned16(m_next)), MGCN_ERR_ALIGN);
  LayerFwdArgs a{};
  a.ns = s; a.nx = x; a.nw = w_in; a.npost = post; a.nhin = (int)Hin;
  a.keep = keep; a.keep_scale = keep_scale;
  a.resid = x_next;   // row-local mode with a finished residual term: the tail reads it from the tile, never from here
  a.res_w = res_w; a.res_b = res_b; a.w_next = w_next; a.pre = pre; a.out_scale = out_scale;
  a.bias = bias;
  a.x_next = x_next; a.m_next = m_next; a.hmask = hmask;
  a.n_rows = N;
  a.act_out = act_out;
  if (w_next == nullptr) {   // no following transform: the streaming pass
    int64_t sb = ceil_div(N, 64);
    if (sb > (int64_t)kNumSMs * 8) sb = (int64_t)kNumSMs * 8;
    MGCN_LAUNCH(k_first_layer_fwd_stream, (unsigned)sb, 256, 0, stream, a);
    return MGCN_OK;
  }
  const size_t smem = sizeof(float) * kFwdSmemFloats;
  // the attribute belongs to (function, device): set on every call (cheap), so a second GPU in the same process
  // gets it too and a failure is reported every time
  cudaError_t attr_err = cudaSuccess;
  {
    attr_err = cudaFuncSetAttribute(k_first_layer_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  MGCN_CHECK_CUDA(attr_err);
  int64_t blocks = ceil_div(ceil_div(N, 16), kFwdWarps);
  if (blocks > (int64_t)kNumSMs * 4) blocks = (int64_t)kNumSMs * 4;
  MGCN_LAUNCH(k_first_layer_fwd, (unsigned)blocks, kFwdWarps * 32, smem, stream, a);
  return MGCN_OK;
}

extern "C" int mgcn_gcn_layer_bwd(const float* dxw, const float* gy, const float* x, const float* w,
                                  const float* res_w, const uint32_t* hmask_prev, const float* post,
                                  int64_t N, int64_t H, float* gy_prev, float* gs_prev, float* dw,
                                  float* d_res_w, float* d_res_b, void* workspace,
                                  size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H == kH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N >= 0 && N < (int64_t(1) << 31), MGCN_ERR_RANGE);
  const int P = bwd_grid(N);
  WorkspaceCarver ws(workspace);
  float* part_w = ws.take<float>((size_t)P * kH * kH);
  float* part_r = ws.take<float>((size_t)P * kH * kH);
  float* part_b = ws.take<float>((size_t)P * kH);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(dxw && gy && x && w && res_w && dw && d_res_w && d_res_b, MGCN_ERR_NULL);
  MGCN_REQUIRE((gy_prev == nullptr) == (gs_prev == nullptr), MGCN_ERR_NULL);
  MGCN_REQUIRE(!gy_prev || hmask_prev, MGCN_ERR_NULL);
  MGCN_REQUIRE(aligned16(dxw) && aligned16(gy) && aligned16(x) && (!gy_prev || aligned16(gy_prev)) &&
                   (!gs_prev || aligned16(gs_prev)),
               MGCN_ERR_ALIGN);
  if (N == 0) return MGCN_OK;
  LayerBwdArgs a{};
  a.dxw = dxw; a.gy = gy; a.x = x; a.w = w; a.res_w = res_w; a.hmask_prev = hmask_prev; a.post = post;
  a.gy_prev = gy_prev; a.gs_prev = gs_prev;
  a.part_w = part_w; a.part_r = part_r; a.part_b = part_b;
  a.n_rows = N;
  const size_t smem = sizeof(float) * kBwdSmemFloats;
  // the attribute belongs to (function, device): set on every call (cheap), so a second GPU in the same process
  // gets it too and a failure is reported every time
  cudaError_t attr_err = cudaSuccess;
  {
    attr_err = cudaFuncSetAttribute(k_layer_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  MGCN_CHECK_CUDA(attr_err);
  MGCN_LAUNCH(k_layer_bwd, P, kBwdWarps * 32, smem, stream, a);
  int rc = launch_reduce_partials(part_w, P, kH * kH, kH, dw, kH, 1, stream);
  if (rc == MGCN_OK) rc = launch_reduce_partials(part_r, P, kH * kH, kH, d_res_w, kH, 1, stream);
  if (rc == MGCN_OK) rc = launch_reduce_partials(part_b, P, kH, kH, d_res_b, 0, 1, stream);
  return rc;
}

// Same contract on tcgen05 / TMEM (gcn_layer_tc.cu).  Measured 0.99 ms against 0.83 ms for the mma.sync
// kernel above at the botnet batch (profiles/r1_layer_summary.md): correct, not yet the default.
extern "C" int mgcn_gcn_layer_bwd_tc(const float* dxw, const float* gy, const float* x, const float* x_scale,
                                     const float* w, const float* res_w, const uint32_t* hmask_prev, const float* post,
                                     int64_t N, int64_t H, float* gy_prev, float* gs_prev, float* dw,
                                     float* d_res_w, float* d_res_b, void* workspace,
                                     size_t* workspace_bytes, void* stream) {
  return mgcn_gcn_layer_bwd_tc_ex(dxw, gy, x, x_scale, w, res_w, hmask_prev, nullptr, post, 1.f, N, H, gy_prev, gs_prev,
                                  dw, d_res_w, d_res_b, nullptr, workspace, workspace_bytes, stream);
}

// + the node-model bias gradient d_bias = bias_scale * colsum(gy * bits(hmask_cur)), summed by the producer warps next
// to dr and reduced in the same launch (k_layer_bwd_tc<true>); d_bias == NULL: the kernel without it.
extern "C" int mgcn_gcn_layer_bwd_tc_ex(const float* dxw, const float* gy, const float* x, const float* x_scale,
                                        const float* w, const float* res_w, const uint32_t* hmask_prev,
                                        const uint32_t* hmask_cur, const float* post, float bias_scale, int64_t N,
                                        int64_t H, float* gy_prev, float* gs_prev, float* dw, float* d_res_w,
                                        float* d_res_b, float* d_bias, void* workspace, size_t* workspace_bytes,
                                        void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H == kH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N >= 0 && N < (int64_t(1) << 31), MGCN_ERR_RANGE);
  WorkspaceCarver ws(workspace);
  float* tc_ws = ws.take<float>(bwd_tc_workspace_floats(N) + (d_bias ? bwd_tc_bias_workspace_floats(N) : 0));
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(dxw && gy && x && w && res_w && dw && d_res_w && d_res_b, MGCN_ERR_NULL);
  MGCN_REQUIRE(!d_bias || hmask_cur, MGCN_ERR_NULL);
  MGCN_REQUIRE((gy_prev == nullptr) == (gs_prev == nullptr), MGCN_ERR_NULL);
  MGCN_REQUIRE(!gy_prev || hmask_prev, MGCN_ERR_NULL);
  MGCN_REQUIRE(aligned16(dxw) && aligned16(gy) && aligned16(x) && (!gy_prev || aligned16(gy_prev)) &&
                   (!gs_prev || aligned16(gs_prev)),
               MGCN_ERR_ALIGN);
  if (N == 0) return MGCN_OK;
  return launch_layer_bwd_tc(dxw, gy, x, x_scale, w, res_w, hmask_prev, post, N, gy_prev, gs_prev, dw, d_res_w,
                             d_res_b, tc_ws, stream, hmask_cur, bias_scale, d_bias);
}

extern "C" int mgcn_mask_bits_scale(const float* gy, const uint32_t* bits, const float* post,
                                    int64_t N, int64_t H, float* gs, void* stream) {
  MGCN_REQUIRE(H == kH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N >= 0 && N < (int64_t(1) << 31), MGCN_ERR_RANGE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(gy && bits && gs, MGCN_ERR_NULL);
  MGCN_REQUIRE(aligned16(gy) && aligned16(gs), MGCN_ERR_ALIGN);
  int64_t blocks = ceil_div(N * (kH / 4), 256);
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  MGCN_LAUNCH(k_mask_bits_scale, (unsigned)blocks, 256, 0, stream, gy, bits, post, N, gs);
  return MGCN_OK;
}

// d_bias[c] = scale * sum_i bit c of bits[i] * gy[i][c]: the bias gradient of a layer without a row-local launch
extern "C" int mgcn_mask_bits_colsum(const float* gy, const uint32_t* bits, float scale, int64_t N, int64_t H,
                                     float* d_bias, void* workspace, size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H == kH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(N >= 0 && N < (int64_t(1) << 31), MGCN_ERR_RANGE);
  WorkspaceCarver ws(workspace);
  float* part = ws.take<float>(mask_bits_colsum_workspace_floats(N));
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(d_bias && (N == 0 || (gy && bits)), MGCN_ERR_NULL);
  MGCN_REQUIRE(aligned16(gy), MGCN_ERR_ALIGN);
  return launch_mask_bits_colsum(gy, bits, scale, N, d_bias, part, stream);   // N == 0: zeros
}
