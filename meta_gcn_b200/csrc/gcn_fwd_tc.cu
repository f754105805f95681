// Forward of one residual GCN layer at hidden 32, AGGREGATE-THEN-TRANSFORM, on the 5th-generation tensor cores
// (gcn_model.py:89-106 around NodeModelAdditive.forward, gcn_base_models.py:199-243):
//
//     s_i  = post_i * sum_{e: col[e]=i} z[row[e]]            z = in_scale (.) x_n   (rows carry the per-source factor)
//     h_i  = relu(s_i W_n + bias)                            hmask_i = bits(h_i > 0)
//     y_i  = h_i + (z_i R_n^T) / in_scale_i + r_n            = h_i + x_i R_n^T + r_n
//     z'_i = out_scale_i * act(y_i)                          act = ReLU, identity for the last layer
//
// (A_hat x) W instead of A_hat (x W): the layer reads ONE [N,32] array (gathered and row-local, the same rows) and
// writes ONE — no message array m = pre (.) (x W) beside x as in k_layer_fwd (gcn_layer.cu), half its DRAM bytes.
// The degree factor of the source travels with the stored rows (z = pre (.) x); the row-local terms undo it with a
// per-row scalar in the epilogue (a row scale commutes with the products), so the gather needs no per-edge weight.
//
// One persistent CTA per SM, 24 warps (80 registers: 6 warps per scheduler) in two roles over 128-row tiles of the work
// order (mgcn_csr_t::tasks):
//   producers  20 warps; a pass = 8 consecutive tasks, one per 4-lane group (gather.cuh: 4 lanes x LDG.256 per
//              gathered row, sums in edge_index order).  The finished sum s and the row's own z are split into tf32
//              hi / lo and stored into SWIZZLE_128B K-major operand images (conflict-free: the 8 lanes of a quarter
//              warp hit 8 different 16-byte bank groups).  Hub segments store their partial sums to the workspace.
//              The warp whose pass completes a tile (16th arrival on the stage's counter, acquire / release) issues
//              the tile's 16 tcgen05.mma (M = 128, K = 8) from one lane:  D1 = s W (main | corrections), D2 = z R^T
//              (main | corrections), 3xTF32 with the correction terms in their own TMEM columns — no issuer warp
//              (a 25th warp would cost every warp 8 registers: 7 warps on one scheduler).
//              Tiles are filled in COMPLETION order: a finished pass takes the next free 8-row slot of the CTA (a
//              shared counter), whatever its place in the work order — a tile of 64-entry rows or hub segments takes
//              16 gather rounds, its neighbours one or two, and with tiles bound to the work order every warp ended
//              up waiting for the slowest pass of the tile two stages back (ncu: a quarter of all instructions were
//              barrier polls).  A row's result does not depend on which rows share its tile, so results stay fixed.
//              The slot's row ids and per-row scalars travel to the epilogue through shared memory.
//   epilogue   4 warps, thread per row: tcgen05.ld -> scalars, ReLUs, mask word -> a 144-byte staged row -> ONE
//              128-byte cp.async.bulk store per row (the TMA engine, not the LSU, moves the outputs)
//   barriers   full[stage] producers -> issuing warp (16 arrivals), done[tile % 2S] tensor core -> producers + epilogue,
//              tfree[stage] epilogue -> issuing warp.  TWO done barriers per stage: a parity wait cannot tell phase u
//              from phase u + 2, and with 20 warps over 16 passes a warp skips a tile now and then, so with one
//              barrier per stage it could find the barrier two phases ahead of the one it waits for and never return
//              (the first version of this kernel did).  With two, a waiter would have to be 4 S tiles behind for the
//              same confusion, and it never skips two tiles in a row.
// Hub rows (longer than the hub threshold) are finished by a second launch of the same kernel (mode 1): its tiles
// walk the hub list, a whole warp sums a hub's segment partials (8 runs in parallel, fixed combine order).
#include <mutex>

#include "common.cuh"
#include "gather.cuh"
#include "tc05.cuh"

namespace mgcn {

constexpr int kFtRows = 128;                     // rows per tile = M of the accumulators
constexpr int kFtImg = kFtRows * 128;            // one operand image: 128 rows x 128 bytes
constexpr int kFtStageB = 4 * kFtImg;            // S_hi, S_lo, Z_hi, Z_lo
#ifndef MGCN_FT_STAGES
#define MGCN_FT_STAGES 2
#endif
constexpr int kFtStages = MGCN_FT_STAGES;   // operand stages == accumulator buffers
constexpr int kFtOffB1 = kFtStages * kFtStageB;  // B1(n, k) = W[k][n]: rows 0..31 hi, 32..63 lo; 64 rows x 128 bytes
constexpr int kFtOffB2 = kFtOffB1 + 8192;        // B2(n, k) = R[n][k]
constexpr int kFtLdo = kFtStages >= 3 ? 32 : 36;   // floats per staged output row: 144-byte rows are conflict-free; with
                                                 // three operand stages only unpadded rows fit (8-way conflicts on the
                                                 // epilogue's 8 stores per row — 3 % of the kernel's wavefronts)
constexpr int kFtOffOut = kFtOffB2 + 8192;
constexpr int kFtOffVec = kFtOffOut + kFtRows * kFtLdo * 4;   // res_b[32], bias[32]
constexpr int kFtOffScal = kFtOffVec + 256;                   // [tile % 2S][128] {post, 1 / in_scale, out_scale, row id}
constexpr int kFtOffMisc = kFtOffScal + 2 * kFtStages * kFtRows * 16;   // barriers, counters, tmem slot
constexpr int kFtSmem = kFtOffMisc + 256 + 1024;
constexpr int kFtEpiWarps = 4;
#ifndef MGCN_FT_PROD
#define MGCN_FT_PROD 20
#endif
constexpr int kFtProdWarps = MGCN_FT_PROD;
constexpr int kFtThreads = 32 * (kFtEpiWarps + kFtProdWarps);
constexpr int kFtTmemCols = kFtStages <= 2 ? 256 : 512;   // accumulator buffers x (D1 main | D1 corr | D2 main | D2 corr)
static_assert(kFtStages >= 2 && kFtStages <= 4, "stages");
static_assert(kFtSmem <= 232448, "shared memory");

struct FwdTcArgs {
  const int4* tasks;
  const int32_t* nbr_w;
  const int32_t* seg_count;
  const int32_t* hub_rows;
  const int32_t* hub_seg0;
  const int32_t* hub_count;
  const int32_t* rowptr;
  const float* z;           // [n_in, 32]
  const float* w;           // weight_node [32 in][32 out]
  const float* res_w;       // residual Linear.weight [32 out][32 in]
  const float* res_b;       // [32] or NULL
  const float* bias;        // node-model bias [32] or NULL
  const float* in_scale;    // [N] or NULL
  const float* post;        // [N] or NULL
  const float* out_scale;   // [N] or NULL
  const uint32_t* keep;     // [N] dropout keep bits of this layer, or NULL (no dropout)
  float keep_scale;         // 1 / (1 - p)
  float* z_next;            // [N, 32]
  uint32_t* hmask;          // [N]
  float* partial;           // [seg_cap, 32]
  int64_t n_rows;
  int64_t seg_cap;
  int64_t hub_cap;
  int act_out;
  int hub_threshold;
};

__device__ __forceinline__ int sw128_off(int r, int q) {   // bytes; 16-byte chunk q of row r, SWIZZLE_128B K-major
  return (r << 7) + ((q ^ (r & 7)) << 4);
}

__device__ __forceinline__ void ft_split4(float a, float b, float c, float d, float4& hi, float4& lo) {
  const float e[4] = {a, b, c, d};
  float h[4], l[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    h[t] = __uint_as_float(round_tf32_bits(__float_as_uint(e[t])));
    l[t] = __uint_as_float(round_tf32_bits(__float_as_uint(e[t] - h[t])));
  }
  hi = make_float4(h[0], h[1], h[2], h[3]);
  lo = make_float4(l[0], l[1], l[2], l[3]);
}

// one row piece (8 columns of this lane) -> hi / lo images at chunks 2 sub, 2 sub + 1 of row r
__device__ __forceinline__ void ft_store_row(unsigned char* img_hi, unsigned char* img_lo, int r, int sub, const Row8& v) {
  float4 hi, lo;
  const int o0 = sw128_off(r, 2 * sub), o1 = sw128_off(r, 2 * sub + 1);
  ft_split4(v.v[0], v.v[1], v.v[2], v.v[3], hi, lo);
  *reinterpret_cast<float4*>(img_hi + o0) = hi;
  *reinterpret_cast<float4*>(img_lo + o0) = lo;
  ft_split4(v.v[4], v.v[5], v.v[6], v.v[7], hi, lo);
  *reinterpret_cast<float4*>(img_hi + o1) = hi;
  *reinterpret_cast<float4*>(img_lo + o1) = lo;
}

__device__ __forceinline__ void ft_tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}

template <int kMode>   // 0: tiles of the work order (rows + hub segments), 1: tiles of the hub list
__global__ void __launch_bounds__(kFtThreads, 1) k_gcn_fwd_tc(const FwdTcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bar_done = reinterpret_cast<uint64_t*>(smem + kFtOffMisc);      // [2 S]: tile tl of this CTA commits to tl % 2S
  uint64_t* bar_tfree = bar_done + 2 * kFtStages;                            // [S]
  uint64_t* bar_full = bar_tfree + kFtStages;                                // [2 S] 16 pass arrivals per tile
  uint32_t* arrivals = reinterpret_cast<uint32_t*>(bar_full + 2 * kFtStages);   // [S] passes stored, never reset
  uint32_t* next_slot = arrivals + kFtStages;                                // passes finished by this CTA so far
  uint32_t* tmem_slot = next_slot + 1;
  float4* scal = reinterpret_cast<float4*>(smem + kFtOffScal);
  float* vec = reinterpret_cast<float*>(smem + kFtOffVec);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

  // weight images (SWIZZLE_128B K-major, 64 rows: hi then lo)
  for (int i = tid; i < 32 * 32; i += kFtThreads) {
    const int n = i >> 5, k = i & 31;
    const float w1 = __ldg(a.w + k * 32 + n), w2 = __ldg(a.res_w + n * 32 + k);
    const float h1 = __uint_as_float(round_tf32_bits(__float_as_uint(w1)));
    const float h2 = __uint_as_float(round_tf32_bits(__float_as_uint(w2)));
    float* b1 = reinterpret_cast<float*>(smem + kFtOffB1);
    float* b2 = reinterpret_cast<float*>(smem + kFtOffB2);
    const int o_hi = (sw128_off(n, k >> 2) >> 2) + (k & 3), o_lo = (sw128_off(n + 32, k >> 2) >> 2) + (k & 3);
    b1[o_hi] = h1;
    b1[o_lo] = __uint_as_float(round_tf32_bits(__float_as_uint(w1 - h1)));
    b2[o_hi] = h2;
    b2[o_lo] = __uint_as_float(round_tf32_bits(__float_as_uint(w2 - h2)));
  }
  if (tid < 32) {
    vec[tid] = a.res_b ? __ldg(a.res_b + tid) : 0.f;
    vec[32 + tid] = a.bias ? __ldg(a.bias + tid) : 0.f;
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kFtStages; ++s) {
      arrivals[s] = 0;
      if (s == 0) *next_slot = 0;
      mbar_init(bar_done + s, 1);
      mbar_init(bar_done + kFtStages + s, 1);
      mbar_init(bar_tfree + s, kFtEpiWarps);
      mbar_init(bar_full + s, 16);
      mbar_init(bar_full + kFtStages + s, 16);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(kFtTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;
  const uint64_t pol = policy_evict_first();

  int64_t limit;   // valid tile entries: tasks (mode 0) or hub rows (mode 1)
  if (kMode == 0) {
    int64_t nseg = 0;
    if (a.seg_count) {
      nseg = *a.seg_count;
      if (nseg > a.seg_cap) nseg = a.seg_cap;
    }
    limit = a.n_rows + nseg;
  } else {
    limit = *a.hub_count;
    if (limit > a.hub_cap) limit = a.hub_cap;
  }
  const int64_t n_tiles = (limit + kFtRows - 1) / kFtRows;

  if (warp >= kFtEpiWarps) {
    // ------------------------------- producers -------------------------------
    const int pw = warp - kFtEpiWarps;
    const uint32_t id64 = umma_idesc_tf32(kFtRows, 64), id32 = umma_idesc_tf32(kFtRows, 32);
    const uint64_t dsc = umma_desc(smem_u32(smem), 16, 1024, 2);   // SWIZZLE_128B K-major: SBO = 8 rows x 128 bytes
    const int sub = lane & 3, grp = lane >> 2, grp_lane0 = grp * 4;
    const unsigned gmask = 0xfu << grp_lane0;
    const int col = sub * 8;
    // descriptors of pass g: lanes 0..7 hold one entry each
    auto load_desc = [&](int64_t g) {
      int4 d = make_int4(-1, 0, 0, 0);
      const int64_t tile = blockIdx.x + (g >> 4) * (int64_t)gridDim.x;
      const int64_t e = tile * kFtRows + (g & 15) * 8 + lane;
      if (lane < 8 && tile < n_tiles && e < limit) {
        if (kMode == 0) {
          d = ld_i4_hint(a.tasks + e, pol);
        } else {
          const int row = __ldg(a.hub_rows + e);
          const int len = __ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row);
          d = make_int4(row, __ldg(a.hub_seg0 + e), (len + a.hub_threshold - 1) / a.hub_threshold, 0);
        }
      }
      return d;
    };
    // software pipeline over this warp's passes: descriptors two passes ahead, the first two index batches one pass
    // ahead, so that a pass starts gathering at once (ncu: 21 % of the producers' stall samples sat on these loads)
    struct PassIdx {
      int beg, end, gi, gin;
    };
    auto load_idx = [&](const int4& d) {
      PassIdx p{0, 0, 0, 0};
      if (kMode == 0) {
        p.beg = __shfl_sync(0xffffffffu, d.y, grp);
        p.end = __shfl_sync(0xffffffffu, d.z, grp);
        if (p.beg + sub < p.end) p.gi = ld_i32_hint(a.nbr_w + p.beg + sub, pol);
        if (p.beg + 4 + sub < p.end) p.gin = ld_i32_hint(a.nbr_w + p.beg + 4 + sub, pol);
      }
      return p;
    };
    int4 d = load_desc(pw);
    int4 dn = load_desc(pw + kFtProdWarps);
    PassIdx pi = load_idx(d);
    // this CTA's tiles of the work order: blockIdx.x, + gridDim.x, ...; its passes fill ceil(passes / 16) tiles
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    for (int64_t g = pw; g < my_tiles * 16; g += kFtProdWarps) {
      const int rowp = __shfl_sync(0xffffffffu, d.x, grp);
      const int slot = __shfl_sync(0xffffffffu, d.w, grp);
      const bool finish = rowp >= 0 && slot == 0;   // this group completes a row
      // the row's own z (unconditional address: the value is only looked at when the row is stored, so the load
      // stays in flight during the gather) and its scalars, one per lane of the group
      const Row8 zrow = ld_row8(a.z + (int64_t)(finish ? rowp : 0) * kGH + col);
      float sc = 1.f;
      {
        const float* sp = sub == 0 ? a.post : sub == 1 ? a.in_scale : sub == 2 ? a.out_scale : nullptr;
        if (finish && sp) sc = __ldg(sp + rowp);   // one load per lane, looked at only when the row is stored
      }
      const PassIdx pc = pi;
      const int4 dc = d;
      d = dn;
      pi = load_idx(d);                               // next pass: index batches in flight during this gather
      dn = load_desc(g + 2 * kFtProdWarps);
      Row8 acc;
#pragma unroll
      for (int q = 0; q < 8; ++q) acc.v[q] = 0.f;
      if (kMode == 0) {
        if (rowp >= 0) {
          acc = gather_sum(a.z, a.nbr_w, pc.beg, pc.end, pc.gi, pc.gin, sub, grp_lane0, gmask, col, pol);
          if (slot != 0) store_partial(a.partial, slot, col, acc);
        }
        // first round of the NEXT pass: its index batch was fetched before this gather and has arrived by now
        if (pi.beg + sub < pi.end) prefetch_row_l2(a.z + (int64_t)pi.gi * kGH);
      } else {
        // the whole warp sums one hub row at a time: 8 contiguous runs of its segment partials in parallel, the run
        // sums added left to right (a fixed order)
#pragma unroll 1
        for (int i = 0; i < 8; ++i) {
          const int rowi = __shfl_sync(0xffffffffu, dc.x, i);
          if (rowi < 0) continue;
          const int s0 = __shfl_sync(0xffffffffu, dc.y, i), ns = __shfl_sync(0xffffffffu, dc.z, i);
          const int per = (ns + 7) >> 3;
          const Row8 run = hub_run_sum(a.partial, s0, grp * per, min(ns, grp * per + per), col);
          Row8 tot;
#pragma unroll
          for (int q = 0; q < 8; ++q) tot.v[q] = __shfl_sync(0xffffffffu, run.v[q], sub);
#pragma unroll
          for (int g2 = 1; g2 < 8; ++g2) {
            Row8 other;
#pragma unroll
            for (int q = 0; q < 8; ++q) other.v[q] = __shfl_sync(0xffffffffu, run.v[q], 4 * g2 + sub);
            if (g2 * per < ns) row8_add(tot, other);
          }
          if (grp == i) acc = tot;
        }
      }
      // next free 8-row slot of this CTA: tile tl (in completion order), rows 8 ps .. 8 ps + 7
      uint32_t my = 0;
      if (lane == 0) asm volatile("atom.relaxed.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(my) : "r"(smem_u32(next_slot)) : "memory");
      my = __shfl_sync(0xffffffffu, my, 0);
      const int64_t tl = my >> 4;
      const int ps = (int)(my & 15u), stage = (int)(tl % kFtStages);
      // the tensor core has consumed this stage's previous tile (tile tl - S of this CTA)
      if (tl >= kFtStages) {
        const int64_t tp = tl - kFtStages;
        mbar_wait(bar_done + (int)(tp % (2 * kFtStages)), (uint32_t)(tp / (2 * kFtStages)) & 1u);
      }
      {
        const int r = ps * 8 + grp;
        if (finish) {
          unsigned char* st = smem + stage * kFtStageB;
          ft_store_row(st, st + kFtImg, r, sub, acc);
          ft_store_row(st + 2 * kFtImg, st + 3 * kFtImg, r, sub, zrow);
        }
        if (sub == 1) sc = __frcp_rn(sc);
        if (sub == 3) sc = __int_as_float(finish ? rowp : -1);
        // slot tl % 2S of the scalar ring: its previous tile tl - 2S was drained by the epilogue before MMA(tl - S)
        // was issued (tfree), and done(tl - S) has just been observed
        reinterpret_cast<float*>(scal + (int)(tl % (2 * kFtStages)) * kFtRows + r)[sub] = sc;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // this lane's image stores -> async proxy
      __syncwarp();
      // arrival: release on the stage's mbarrier; a relaxed counter only elects the warp that issues the tile's MMAs,
      // which then acquires through the mbarrier (16 arrivals) — no acq_rel atomic, no MEMBAR per pass
      uint32_t old = 0;
      if (lane == 0) {
        mbar_arrive(bar_full + (int)(tl % (2 * kFtStages)));
        asm volatile("atom.relaxed.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(arrivals + stage)) : "memory");
      }
      old = __shfl_sync(0xffffffffu, old, 0);
      if ((old & 15u) == 15u) {
        // 16th pass of the tile: wait for the other passes' arrivals (acquire), then the accumulator buffer
        const uint32_t use = (uint32_t)(tl / kFtStages);
        mbar_wait(bar_full + (int)(tl % (2 * kFtStages)), (uint32_t)(tl / (2 * kFtStages)) & 1u);
        if (use >= 1) mbar_wait(bar_tfree + stage, (use - 1) & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (lane == 0) {
          const uint32_t tb = tmem + stage * 128;
          const uint32_t so = (uint32_t)(stage * kFtStageB) >> 4;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t ko = 2 * k;   // 8 tf32 = 32 bytes inside the 128-byte swizzle row
            const uint64_t b1 = dsc + ((kFtOffB1 >> 4) + ko), b2 = dsc + ((kFtOffB2 >> 4) + ko);
            umma_tf32(tb + 0, dsc + (so + ko), b1, id64, k > 0);                          // s_hi [W_hi | W_lo]
            umma_tf32(tb + 32, dsc + (so + (kFtImg >> 4) + ko), b1, id32, 1);             // s_lo W_hi
            umma_tf32(tb + 64, dsc + (so + (2 * kFtImg >> 4) + ko), b2, id64, k > 0);     // z_hi [R_hi | R_lo]
            umma_tf32(tb + 96, dsc + (so + (3 * kFtImg >> 4) + ko), b2, id32, 1);         // z_lo R_hi
          }
          umma_commit(bar_done + (int)(tl % (2 * kFtStages)));
        }
        __syncwarp();
      }
    }
  } else {
    // ------------------------------- epilogue: thread per row -------------------------------
    const int r = 32 * warp + lane;
    float* stg = reinterpret_cast<float*>(smem + kFtOffOut) + r * kFtLdo;
    int tl = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
      const int stage = tl % kFtStages;
      mbar_wait(bar_done + tl % (2 * kFtStages), (uint32_t)(tl / (2 * kFtStages)) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the staged row of the previous tile has been read
      // acquire the producers' scalar / row-id stores (two full barriers per stage, like done: this wait may come
      // after the stage's NEXT tile has filled)
      mbar_wait(bar_full + tl % (2 * kFtStages), (uint32_t)(tl / (2 * kFtStages)) & 1u);
      const float4 sc4 = scal[(tl % (2 * kFtStages)) * kFtRows + r];
      const float postv = sc4.x, inv = sc4.y, outs = sc4.z;
      const int row = __float_as_int(sc4.w);
      const uint32_t kept = (a.keep && row >= 0) ? __ldg(a.keep + row) : 0xffffffffu;
      const uint32_t ta = tmem + stage * 128 + ((uint32_t)(32 * warp) << 16);
      uint32_t bits = 0;
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 8) {
        uint32_t m1[8], c1[8], m2[8], c2[8];
        ft_tmem_ld8(ta + c0, m1);
        ft_tmem_ld8(ta + 32 + c0, c1);
        ft_tmem_ld8(ta + 64 + c0, m2);
        ft_tmem_ld8(ta + 96 + c0, c2);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        float o[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const int c = c0 + t;
          const float v1 = __uint_as_float(m1[t]) + __uint_as_float(c1[t]);
          const float v2 = __uint_as_float(m2[t]) + __uint_as_float(c2[t]);
          float h = __fmul_rn(postv, v1) + vec[32 + c];
          h = h > 0.f ? h : 0.f;
          // dropout: one rounded multiply (no contraction into the add below), as torch's dropout; a dropped entry is
          // one more cleared bit of the ReLU mask word
          if (a.keep) h = ((kept >> c) & 1u) ? __fmul_rn(h, a.keep_scale) : 0.f;
          bits |= (h > 0.f ? 1u : 0u) << c;
          float y = h + (__fmul_rn(inv, v2) + vec[c]);
          if (a.act_out == 1) y = y > 0.f ? y : 0.f;
          o[t] = y * outs;
        }
        *reinterpret_cast<float4*>(stg + c0) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4*>(stg + c0 + 4) = make_float4(o[4], o[5], o[6], o[7]);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tfree + stage);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // staged row -> visible to the bulk copy
      if (row >= 0) {
        a.hmask[row] = bits;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], 128, %2;" ::"l"(
                         a.z_next + (int64_t)row * kGH),
                     "r"(smem_u32(stg)), "l"(pol)
                     : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kFtTmemCols) : "memory");
  }
}

}  // namespace mgcn

using namespace mgcn;

extern "C" int mgcn_gcn_layer_fwd_tc(const mgcn_csr_t* g, const float* z, int64_t n_in, const float* w,
                                     const float* res_w, const float* res_b, const float* bias,
                                     const float* in_scale, const float* post, const float* out_scale, int act_out,
                                     int64_t H, float* z_next, uint32_t* hmask, void* workspace,
                                     size_t* workspace_bytes, void* stream) {
  return mgcn_gcn_layer_fwd_tc_ex(g, z, n_in, w, res_w, res_b, bias, in_scale, post, out_scale, nullptr, 1.f, act_out,
                                  H, z_next, hmask, workspace, workspace_bytes, stream);
}

extern "C" int mgcn_gcn_layer_fwd_tc_ex(const mgcn_csr_t* g, const float* z, int64_t n_in, const float* w,
                                        const float* res_w, const float* res_b, const float* bias,
                                        const float* in_scale, const float* post, const float* out_scale,
                                        const uint32_t* keep, float keep_scale, int act_out, int64_t H, float* z_next,
                                        uint32_t* hmask, void* workspace, size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr && g != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(H == kGH, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(act_out == 0 || act_out == 1, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(n_in >= 0 && g->n_rows >= 0, MGCN_ERR_RANGE);
  const bool hubs = g->hub_rows && g->hub_seg0 && g->hub_count && g->seg_count && g->hub_cap > 0 && g->seg_cap > 0;
  WorkspaceCarver ws(workspace);
  float* partial = ws.take<float>(hubs ? (size_t)g->seg_cap * kGH : 0);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  if (g->n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(z && w && res_w && z_next && hmask && g->rowptr && g->tasks, MGCN_ERR_NULL);
  MGCN_REQUIRE(g->nnz_cap == 0 || g->nbr_w, MGCN_ERR_NULL);
  MGCN_REQUIRE((reinterpret_cast<uintptr_t>(z) & 31u) == 0, MGCN_ERR_ALIGN);   // 256-bit row gathers
  MGCN_REQUIRE(aligned16(g->tasks) && aligned16(z_next) && aligned16(partial), MGCN_ERR_ALIGN);
  FwdTcArgs a{};
  a.tasks = reinterpret_cast<const int4*>(g->tasks);
  a.nbr_w = g->nbr_w;
  a.seg_count = hubs ? g->seg_count : nullptr;
  a.hub_rows = g->hub_rows;
  a.hub_seg0 = g->hub_seg0;
  a.hub_count = g->hub_count;
  a.rowptr = g->rowptr;
  a.hub_threshold = g->hub_threshold;
  a.z = z; a.w = w; a.res_w = res_w; a.res_b = res_b; a.bias = bias;
  a.in_scale = in_scale; a.post = post; a.out_scale = out_scale;
  a.keep = keep; a.keep_scale = keep_scale;
  a.z_next = z_next; a.hmask = hmask; a.partial = partial;
  a.n_rows = g->n_rows;
  a.seg_cap = hubs ? g->seg_cap : 0;
  a.hub_cap = hubs ? g->hub_cap : 0;
  a.act_out = act_out;
  int dev = 0, sms = 0;
  MGCN_CHECK_CUDA(cudaGetDevice(&dev));
  MGCN_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  MGCN_CHECK_CUDA(cudaFuncSetAttribute(k_gcn_fwd_tc<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFtSmem));
  MGCN_CHECK_CUDA(cudaFuncSetAttribute(k_gcn_fwd_tc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFtSmem));
  int64_t tiles = ceil_div(a.n_rows + a.seg_cap, kFtRows);
  MGCN_LAUNCH(k_gcn_fwd_tc<0>, (unsigned)(tiles < sms ? tiles : sms), kFtThreads, kFtSmem, stream, a);
  if (hubs) {
    tiles = ceil_div(a.hub_cap, kFtRows);
    MGCN_LAUNCH(k_gcn_fwd_tc<1>, (unsigned)(tiles < sms ? tiles : sms), kFtThreads, kFtSmem, stream, a);
  }
  return MGCN_OK;
}
