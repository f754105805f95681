// Row-local backward of one residual GCN layer at hidden 32 on the 5th-generation tensor cores
// (tcgen05.mma, accumulators in tensor memory), entry points mgcn_gcn_layer_bwd_tc* (gcn_layer.cu):
//     G = dxw W^T + gy R;   dW = x^T dxw;   dR = gy^T x;   dr = colsum(gy)
//     gy_prev = G * (x > 0);   gs_prev = post * gy_prev * bits(hmask_prev)
// Every operand element is split ONCE into hi/lo tf32 images in shared memory and one thread issues 24
// tcgen05.mma per 64-row tile:
//   row-local   D[64 x 64|32] (+)= A_K[64 x 8] * B_K[64|32 x 8]^T        K-major, un-swizzled interleaved images
//               TMEM cols [0,32) main = dxw_hi Wt_hi + gy_hi R_hi; [32,64) = hi * B_lo + lo * B_hi (both corrections)
//               (M = 64 accumulators occupy 16 lanes of each 32-lane TMEM quarter; the D address may start at lane 0
//               or 16, so the two tiles of a pair share one set of columns: tile 2j in lanes 0..15, tile 2j+1 in 16..31)
//   transposed  [D1 | D2][128 x 64] (+)= [dxw_hi|gy_hi|dxw_lo|gy_lo]^T[128 x 8 rows] * [x_hi | x_lo][8 rows x 64]
//               MN-major, SWIZZLE_128B_BASE32B images, TMEM cols [64,128) (tile 2j) and [128,192) (tile 2j+1)
//               rows 0-31 -> dW^T, 32-63 -> dR (main terms), 64-127 -> their corrections
// (a 32-bit MN-major operand is only read correctly from the BASE32B image, a K-major one never from it —
// scripts/tc_probe.cu — hence dxw and gy are stored in both images.)  Chains through the TMEM accumulator
// stay short (8 steps) and start from zero in every tile; sums over tiles are RN adds in registers;
// per-CTA partials are reduced in a fixed order.
//
// One persistent CTA per SM, 24 warps in three roles (k_layer_bwd_tc below):
//   producers  2 sets x 8 warps, set p owns operand stage p (80 KB of images) and the tiles with it % 2 == p:
//              LDG.256 one tile ahead -> split -> 20 conflict-free STS.128 per thread; warp 0 of a set also issues
//              the tile's tcgen05.mma and commits to the stage's `done` barrier
//   epilogue   8 warps (TMEM quarter = warp % 4, column half = warp / 4) work on tile PAIRS: all 32 lanes carry a
//              G row, outputs are staged in shared memory (144-byte rows) and leave as whole 512-byte row groups
//   barriers   full[stage] producers -> issuer, done[pair buffer][set] tensor core -> producers + epilogue,
//              tfree[pair buffer] epilogue -> issuers   (done is per pair buffer so that no waiter can be lapped)
// Measured at the botnet batch (profiles/r1b_layer_summary.md): 0.99 ms as CTA-wide phases -> 0.58 ms, against 0.81 ms
// for the mma.sync kernel it replaced; 4.0 TB/s of algorithmic bytes.  The limiter is now the shared-memory data pipe
// (l1tex__data_pipe_lsu_wavefronts 83 %: 47 M store wavefronts for the ten images + the tensor core's operand
// reads), not HBM (48 %) or the tensor pipe (23 %).
#include <mutex>

#include "common.cuh"
#include "tc05.cuh"

namespace mgcn {

constexpr int kTH = 32;
constexpr int kTRows = 64;                 // rows per tile (M = 64 accumulators; two operand stages of 80 KB fit one SM)
constexpr int kTileB = kTRows * kTH * 4;   // 8 KB per image

struct BwdTcArgs {
  const float* dxw;
  const float* gy;
  const float* x;
  const float* x_scale;      // [N] or NULL: the stored rows are x_scale (.) x (aggregate-then-transform stack); undone on load
  const float* w;            // weight_node (in j, out c)
  const float* res_w;        // residual weight (out c, in j)
  const uint32_t* hmask_prev;
  const float* post;
  float* gy_prev;
  float* gs_prev;
  float* part_t;             // [grid][128][32]
  float* part_b;             // [grid][32]
  int64_t n_rows;
};

// shared-memory map (bytes from a 1024-aligned base); one operand stage = 10 images = 80 KB
constexpr int kOffKDh = 0;                 // K-major images of dxw_hi, dxw_lo, gy_hi, gy_lo
constexpr int kOffKDl = 1 * kTileB;
constexpr int kOffKGh = 2 * kTileB;
constexpr int kOffKGl = 3 * kTileB;
constexpr int kOffMN = 4 * kTileB;         // MN-major images [dxw_hi | gy_hi | dxw_lo | gy_lo]
constexpr int kOffMXh = 8 * kTileB;        // MN-major x_hi, x_lo
constexpr int kOffMXl = 9 * kTileB;
constexpr int kStageB = 10 * kTileB;
constexpr int kStages = 2;                 // operand stages == TMEM accumulator buffers
constexpr int kOffB1 = kStages * kStageB;  // [Wt_hi ; Wt_lo]  64 x 32, K-major
constexpr int kOffB2 = kOffB1 + 8192;      // [R_hi ; R_lo]
constexpr int kOffMisc = kOffB2 + 8192;    // barriers (full[2], done[2], tfree[2]), tmem slot
constexpr int kOffXbits = kOffMisc + 128;   // [8][64] words: x > 0 of the tile's rows (8 tiles deep)
constexpr int kLdo = 36;                   // floats per staged output row (144 bytes)
constexpr int kOffOut = kOffXbits + 8 * 64 * 4;     // [2 tiles of a pair][gy_prev | gs_prev][64 rows][kLdo] staged outputs
constexpr int kOffDrRed = kOffOut + 2 * 2 * kTRows * kLdo * 4;   // [16 producer warps][32] dr partials
constexpr int kBwdTcSmem = kOffDrRed + 16 * 32 * 4 + 1024;
constexpr int kTmemBufCols = 256;          // accumulator columns per pair buffer: G main [0,32) and corrections [32,64) of both
                                           // tiles (tile 2j in lanes 0..15, tile 2j+1 in lanes 16..31 of every quarter),
                                           // transposed products of tile 2j [64,128) and of tile 2j+1 [128,192)

constexpr int kEpiWarps = 8;               // warps 0..7   TMEM -> registers -> gy_prev / gs_prev, running dW / dR rows
constexpr int kProdWarps = 16;             // warps 8..23  global -> split -> operand images (two sets of 8, one per stage)
constexpr int kBwdTcThreads = 32 * (kEpiWarps + kProdWarps);       // warp 0 of a producer set issues its tcgen05.mma

__device__ __forceinline__ int k_image_off(int r, int q) {      // bytes; 16-byte chunk q of row r, interleaved
  return ((r >> 3) << 10) + (q << 7) + ((r & 7) << 4);
}
__device__ __forceinline__ int mn_image_off(int r, int q) {     // bytes; SWIZZLE_128B_BASE32B
  return (r << 7) + ((((q >> 1) ^ (r & 3)) << 5) | ((q & 1) << 4));
}

__device__ __forceinline__ void split4(const float4 v, float4& hi, float4& lo) {
  const float e[4] = {v.x, v.y, v.z, v.w};
  float h[4], l[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    h[t] = __uint_as_float(round_tf32_bits(__float_as_uint(e[t])));
    l[t] = __uint_as_float(round_tf32_bits(__float_as_uint(e[t] - h[t])));
  }
  hi = make_float4(h[0], h[1], h[2], h[3]);
  lo = make_float4(l[0], l[1], l[2], l[3]);
}

struct F8 {
  float4 lo, hi;
};
__device__ __forceinline__ F8 ld_f8_hint(const float* p, uint64_t pol) {   // one LDG.256, streamed
  F8 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
               : "=f"(r.lo.x), "=f"(r.lo.y), "=f"(r.lo.z), "=f"(r.lo.w), "=f"(r.hi.x), "=f"(r.hi.y), "=f"(r.hi.z), "=f"(r.hi.w)
               : "l"(p), "l"(pol));
  return r;
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}

// Warp-specialised, one persistent CTA per SM.  Tile `it` of a CTA uses operand stage / accumulator buffer
// s = it & 1 for the (it >> 1)-th time; three mbarriers per stage carry the hand-offs:
//   full[s]   producers -> MMA warp        the 10 images of the tile are written (8 arrivals, one per warp)
//   done[s]   tensor core -> everyone      tcgen05.commit: accumulators ready, images free again
//   tfree[s]  epilogue -> MMA warp         accumulator buffer s has been read (8 arrivals)
// so the split of tile it+1, the tensor-core work of tile it+1 and the epilogue of tile it overlap.
__global__ void __launch_bounds__(kBwdTcThreads, 1) k_layer_bwd_tc(const BwdTcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // 1024-byte alignment as an offset on the __shared__ array (keeps the shared address space: STS, not ST)
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + kOffMisc);
  uint64_t* bar_done = bar_full + 2;
  uint64_t* bar_tfree = bar_full + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffMisc + 80);
  uint32_t* xbits = reinterpret_cast<uint32_t*>(smem + kOffXbits);
  float* dr_red = reinterpret_cast<float*>(smem + kOffDrRed);   // [16 warps][32]
  float* stage_out = reinterpret_cast<float*>(smem + kOffOut);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler (roles, descriptors)
  const bool want_prev = a.gy_prev != nullptr;

  // weight images: B1(n, k) = W[n][k] (hi rows 0..31, lo rows 32..63); B2(n, k) = R[k][n]
  for (int i = tid; i < 32 * 32; i += kBwdTcThreads) {
    const int n = i >> 5, k = i & 31;
    const float w1 = __ldg(a.w + n * 32 + k), w2 = __ldg(a.res_w + k * 32 + n);
    const float h1 = __uint_as_float(round_tf32_bits(__float_as_uint(w1)));
    const float h2 = __uint_as_float(round_tf32_bits(__float_as_uint(w2)));
    float* b1 = reinterpret_cast<float*>(smem + kOffB1);
    float* b2 = reinterpret_cast<float*>(smem + kOffB2);
    const int o_hi = (k_image_off(n, k >> 2) >> 2) + (k & 3), o_lo = (k_image_off(n + 32, k >> 2) >> 2) + (k & 3);
    b1[o_hi] = h1;
    b1[o_lo] = __uint_as_float(round_tf32_bits(__float_as_uint(w1 - h1)));
    b2[o_hi] = h2;
    b2[o_lo] = __uint_as_float(round_tf32_bits(__float_as_uint(w2 - h2)));
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full + s, kProdWarps / 2);
      mbar_init(bar_done + s, 1);
      mbar_init(bar_done + 2 + s, 1);
      mbar_init(bar_tfree + s, kEpiWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // weight images -> visible to the tensor core
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;
  const uint64_t pol = policy_evict_first();
  const int64_t n_tiles = (a.n_rows + kTRows - 1) / kTRows;

  if (warp >= kEpiWarps && warp < kEpiWarps + kProdWarps) {
    // ---------------- producers: global -> registers (one tile ahead) -> hi/lo split -> images ----------------
    // Two sets of 8 warps: set p produces the tiles with it % 2 == p, i.e. always into stage p, so a set has
    // two tile periods for one tile.  Lane 8 qq + j of warp w owns row 8 w + j and the 32-byte chunk pair qq
    // (one LDG.256 per array); the two 16-byte chunks are stored in the order (j >> 2) ? (hi, lo) : (lo, hi) so
    // that the 8 lanes of a quarter warp hit 8 different 16-byte bank groups in the K-major images (bank group
    // = row & 7) and in the swizzled MN-major ones (bank group = (((q >> 1) ^ (row & 3)) << 1) | (q & 1)).
    const int pset = (warp - kEpiWarps) >> 3, pwarp = (warp - kEpiWarps) & 7;
    const int j = lane & 7, qq = lane >> 3, flip = j >> 2;
    const int r0 = 8 * pwarp + j;
    const int qa = 2 * qq + flip, qb = 2 * qq + (flip ^ 1);
    const int ko_a = k_image_off(r0, qa), ko_b = k_image_off(r0, qb);
    const int mo_a = mn_image_off(r0, qa), mo_b = mn_image_off(r0, qb);
    float acc_dr[2][4];   // column sums of gy over this thread's rows
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int t = 0; t < 4; ++t) acc_dr[i][t] = 0.f;
    F8 cur[3], nxt[3];
    float xs_cur = 1.f, xs_nxt = 1.f;   // 1 / x_scale of this thread's row, fetched with the tile, applied at use
    auto load_tile = [&](F8 (&dst)[3], float& xs_out, int64_t tile) {
      const float* src[3] = {a.dxw, a.gy, a.x};
      const int64_t gr = tile * kTRows + r0;
      const bool ok = tile < n_tiles && gr < a.n_rows;
      xs_out = 1.f;
      if (ok && a.x_scale) xs_out = __ldg(a.x_scale + gr);
#pragma unroll
      for (int arr = 0; arr < 3; ++arr) {
        F8 v;
        v.lo = v.hi = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) v = ld_f8_hint(src[arr] + gr * kTH + 8 * qq, pol);
        dst[arr] = v;
      }
    };
    unsigned char* st = smem + pset * kStageB;
    const uint32_t idG64 = umma_idesc_tf32(64, 64), idG32 = umma_idesc_tf32(64, 32), idT = umma_idesc_tf32(128, 64, 1, 1);
    // descriptor templates: the start-address field (bits 0..13, 16-byte units) is added per stage and k step
    const uint64_t dK = umma_desc(smem_u32(smem), 128, 1024, 0), dM = umma_desc(smem_u32(smem), kTileB, 512, 1);
    int it = pset;
    int64_t tile = blockIdx.x + (int64_t)pset * gridDim.x;
    load_tile(cur, xs_cur, tile);
    for (; tile < n_tiles; tile += 2 * (int64_t)gridDim.x, it += 2) {
      load_tile(nxt, xs_nxt, tile + 2 * (int64_t)gridDim.x);
      const int use = it >> 1;
      // the tensor core has consumed this stage's previous tile (done barriers: [pair buffer][set])
      if (use >= 1) mbar_wait(bar_done + 2 * ((use - 1) & 1) + pset, ((use - 1) >> 1) & 1);
      float4 c0, c1, hi, lo;
      // dxw
      c0 = flip ? cur[0].hi : cur[0].lo;
      c1 = flip ? cur[0].lo : cur[0].hi;
      split4(c0, hi, lo);
      *reinterpret_cast<float4*>(st + kOffKDh + ko_a) = hi;
      *reinterpret_cast<float4*>(st + kOffKDl + ko_a) = lo;
      *reinterpret_cast<float4*>(st + kOffMN + 0 * kTileB + mo_a) = hi;
      *reinterpret_cast<float4*>(st + kOffMN + 2 * kTileB + mo_a) = lo;
      split4(c1, hi, lo);
      *reinterpret_cast<float4*>(st + kOffKDh + ko_b) = hi;
      *reinterpret_cast<float4*>(st + kOffKDl + ko_b) = lo;
      *reinterpret_cast<float4*>(st + kOffMN + 0 * kTileB + mo_b) = hi;
      *reinterpret_cast<float4*>(st + kOffMN + 2 * kTileB + mo_b) = lo;
      // gy
      {
        const float4 g0 = cur[1].lo, g1 = cur[1].hi;
        acc_dr[0][0] += g0.x; acc_dr[0][1] += g0.y; acc_dr[0][2] += g0.z; acc_dr[0][3] += g0.w;
        acc_dr[1][0] += g1.x; acc_dr[1][1] += g1.y; acc_dr[1][2] += g1.z; acc_dr[1][3] += g1.w;
      }
      c0 = flip ? cur[1].hi : cur[1].lo;
      c1 = flip ? cur[1].lo : cur[1].hi;
      split4(c0, hi, lo);
      *reinterpret_cast<float4*>(st + kOffKGh + ko_a) = hi;
      *reinterpret_cast<float4*>(st + kOffKGl + ko_a) = lo;
      *reinterpret_cast<float4*>(st + kOffMN + 1 * kTileB + mo_a) = hi;
      *reinterpret_cast<float4*>(st + kOffMN + 3 * kTileB + mo_a) = lo;
      split4(c1, hi, lo);
      *reinterpret_cast<float4*>(st + kOffKGh + ko_b) = hi;
      *reinterpret_cast<float4*>(st + kOffKGl + ko_b) = lo;
      *reinterpret_cast<float4*>(st + kOffMN + 1 * kTileB + mo_b) = hi;
      *reinterpret_cast<float4*>(st + kOffMN + 3 * kTileB + mo_b) = lo;
      // x
      if (a.x_scale) {
        const float xs = __frcp_rn(xs_cur);
        F8& v = cur[2];
        v.lo.x *= xs; v.lo.y *= xs; v.lo.z *= xs; v.lo.w *= xs;
        v.hi.x *= xs; v.hi.y *= xs; v.hi.z *= xs; v.hi.w *= xs;
      }
      uint32_t b;
      {
        const float4 x0 = cur[2].lo, x1 = cur[2].hi;
        b = (x0.x > 0.f ? 1u : 0u) | (x0.y > 0.f ? 2u : 0u) | (x0.z > 0.f ? 4u : 0u) | (x0.w > 0.f ? 8u : 0u) |
            (x1.x > 0.f ? 16u : 0u) | (x1.y > 0.f ? 32u : 0u) | (x1.z > 0.f ? 64u : 0u) | (x1.w > 0.f ? 128u : 0u);
        b <<= 8 * qq;
      }
      c0 = flip ? cur[2].hi : cur[2].lo;
      c1 = flip ? cur[2].lo : cur[2].hi;
      split4(c0, hi, lo);
      *reinterpret_cast<float4*>(st + kOffMXh + mo_a) = hi;
      *reinterpret_cast<float4*>(st + kOffMXl + mo_a) = lo;
      split4(c1, hi, lo);
      *reinterpret_cast<float4*>(st + kOffMXh + mo_b) = hi;
      *reinterpret_cast<float4*>(st + kOffMXl + mo_b) = lo;
      b |= __shfl_xor_sync(0xffffffffu, b, 8);
      b |= __shfl_xor_sync(0xffffffffu, b, 16);
      if (qq == 0) xbits[(it & 7) * 64 + r0] = b;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_full + pset);
      if (pwarp == 0) {
        // this warp also issues the tile's 24 tcgen05.mma (lane 0) once the other 7 warps of the set have arrived
        // and the epilogue has drained accumulator buffer pset
        mbar_wait(bar_full + pset, use & 1);
        // pair buffer of tiles (2 use, 2 use + 1): read by the epilogue two pairs ago
        const int pb = use & 1;
        if (use >= 2) mbar_wait(bar_tfree + pb, ((use >> 1) - 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (lane == 0) {
          const uint32_t tb = tmem + pb * kTmemBufCols;
          const uint32_t tg = tb + ((uint32_t)(16 * pset) << 16);   // M = 64 accumulators of this set's tile: lanes 16 pset ..
          const uint32_t tt = tb + 64 + 64 * pset;
          const uint32_t so = (uint32_t)(pset * kStageB) >> 4;
          if (want_prev) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t ko = (256 * k) >> 4;   // 8 columns = two 16-byte chunks
              const uint64_t b1 = dK + ((kOffB1 >> 4) + ko), b2 = dK + ((kOffB2 >> 4) + ko);
              umma_tf32(tg + 0, dK + (so + (kOffKDh >> 4) + ko), b1, idG64, k > 0);    // dxw_hi [Wt_hi | Wt_lo]
              umma_tf32(tg + 0, dK + (so + (kOffKGh >> 4) + ko), b2, idG64, 1);        // gy_hi  [R_hi | R_lo]
              umma_tf32(tg + 32, dK + (so + (kOffKDl >> 4) + ko), b1, idG32, 1);       // dxw_lo Wt_hi  (joins hi * B_lo)
              umma_tf32(tg + 32, dK + (so + (kOffKGl >> 4) + ko), b2, idG32, 1);       // gy_lo  R_hi
            }
          }
#pragma unroll
          for (int k = 0; k < kTRows / 8; ++k) {
            const uint32_t ko = (1024 * k) >> 4;    // 8 rows = two 4-row atoms
            // B = [x_hi | x_lo]: two 32-column MN atoms one image apart -> D1 | D2 in one N = 64 instruction
            umma_tf32(tt, dM + (so + (kOffMN >> 4) + ko), dM + (so + (kOffMXh >> 4) + ko), idT, k > 0);
          }
          umma_commit(bar_done + 2 * pb + pset);
        }
        __syncwarp();
      }
#pragma unroll
      for (int arr = 0; arr < 3; ++arr) cur[arr] = nxt[arr];
      xs_cur = xs_nxt;
    }
    // dr[c]: this thread holds columns 8 qq + 4 i + t summed over its rows; rows of the warp are added in a fixed
    // butterfly order, the 16 warps by one thread per column below
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float v = acc_dr[i][t];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        if (j == 0) dr_red[(warp - kEpiWarps) * 32 + 8 * qq + 4 * i + t] = v;
      }
  } else {
    // ---------------- epilogue warps: quarter = warp & 3 of the TMEM lanes, column half = warp >> 2 ----------------
    const int quarter = warp & 3, half = warp >> 2;
    float acc_t[16];      // running transposed-product row of this TMEM lane, 16 of its 32 columns
#pragma unroll
    for (int t = 0; t < 16; ++t) acc_t[t] = 0.f;
    // tile 2j of a pair lives in lanes 0..15, tile 2j + 1 in lanes 16..31 of every quarter (M = 64 accumulators)
    const int my_row = 16 * quarter + (lane & 15), sel = lane >> 4;
    // mask word and per-target factor of this lane's row, fetched one pair ahead
    uint32_t hbits_n = 0;
    float post_n = 1.f;
    auto load_row_scalars = [&](int64_t tile) {
      const int64_t gr = tile * kTRows + my_row;
      hbits_n = 0;
      post_n = 1.f;
      if (want_prev && tile < n_tiles && gr < a.n_rows) {
        hbits_n = __ldg(a.hmask_prev + gr);
        if (a.post) post_n = __ldg(a.post + gr);
      }
    };
    load_row_scalars(blockIdx.x + (int64_t)sel * gridDim.x);
    int j = 0;
    for (int64_t tile_a = blockIdx.x; tile_a < n_tiles; tile_a += 2 * (int64_t)gridDim.x, ++j) {
      const int pb = j & 1;
      const int64_t tile_b = tile_a + gridDim.x;
      const bool has_b = tile_b < n_tiles;
      const uint32_t hbits = hbits_n;
      const float postv = post_n;
      load_row_scalars(tile_a + (int64_t)(2 + sel) * gridDim.x);
      mbar_wait(bar_done + 2 * pb + 0, (j >> 1) & 1);
      if (has_b) mbar_wait(bar_done + 2 * pb + 1, (j >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t lane_addr = tmem + pb * kTmemBufCols + ((uint32_t)(32 * quarter) << 16);
#pragma unroll
      for (int t2 = 0; t2 < 2; ++t2) {
        if (t2 == 0 || has_b) {
          // transposed products of one tile -> running fp32 sums (RN)
          uint32_t d1[16], d2[16];
          tmem_ld16(lane_addr + 64 + 64 * t2 + 16 * half, d1);
          tmem_ld16(lane_addr + 96 + 64 * t2 + 16 * half, d2);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int t = 0; t < 16; ++t) acc_t[t] += __uint_as_float(d1[t]) + __uint_as_float(d2[t]);
        }
      }
      if (want_prev) {
        // G row of this lane, columns [16 half, 16 half + 16) -> staging tile in shared memory (rows padded to 144
        // bytes: the 8 rows of a quarter warp land in 8 different 16-byte bank groups)
        const uint32_t xb = xbits[((2 * j + sel) & 7) * 64 + my_row];
        float* sg = stage_out + sel * (2 * kTRows * kLdo);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c0 = 16 * half + 8 * h;
          uint32_t m[8], c1[8];
          tmem_ld8(lane_addr + 0 + c0, m);
          tmem_ld8(lane_addr + 32 + c0, c1);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            float g[4], sv[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const int c = c0 + 4 * q + t;
              const float gv = __uint_as_float(m[4 * q + t]) + __uint_as_float(c1[4 * q + t]);
              g[t] = ((xb >> c) & 1u) ? gv : 0.f;
              sv[t] = ((hbits >> c) & 1u) ? g[t] * postv : 0.f;
            }
            *reinterpret_cast<float4*>(sg + my_row * kLdo + c0 + 4 * q) = make_float4(g[0], g[1], g[2], g[3]);
            *reinterpret_cast<float4*>(sg + (kTRows + my_row) * kLdo + c0 + 4 * q) = make_float4(sv[0], sv[1], sv[2], sv[3]);
          }
        }
      }
      // pair buffer pb is free for the pair after next
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tfree + pb);
      if (want_prev) {
        // staged rows -> global, 4 whole rows (512 contiguous bytes) per store instruction; warp w owns rows
        // 8w..8w+7 of both tiles
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
#pragma unroll
        for (int t2 = 0; t2 < 2; ++t2) {
          if (t2 == 0 || has_b) {
            const float* sgo = stage_out + t2 * (2 * kTRows * kLdo);
            const int64_t tile = t2 == 0 ? tile_a : tile_b;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int r = 8 * warp + 4 * i + (lane >> 3), q = lane & 7;
              const int64_t gr = tile * kTRows + r;
              if (gr < a.n_rows) {
                st_f4_hint(a.gy_prev + gr * kTH + 4 * q, *reinterpret_cast<const float4*>(sgo + r * kLdo + 4 * q), pol);
                st_f4_hint(a.gs_prev + gr * kTH + 4 * q, *reinterpret_cast<const float4*>(sgo + (kTRows + r) * kLdo + 4 * q), pol);
              }
            }
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");   // staging tile may be rewritten
      }
    }
    // per-CTA partials of the transposed products: row = TMEM lane, this warp's 16 columns
    float* p = a.part_t + ((int64_t)blockIdx.x * 128 + 32 * quarter + lane) * 32 + 16 * half;
#pragma unroll
    for (int t = 0; t < 16; t += 4) *reinterpret_cast<float4*>(p + t) = make_float4(acc_t[t], acc_t[t + 1], acc_t[t + 2], acc_t[t + 3]);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) {
    float s = 0.f;
    for (int w = 0; w < kProdWarps; ++w) s += dr_red[w * 32 + tid];
    a.part_b[(int64_t)blockIdx.x * 32 + tid] = s;
  }
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
  }
}

// dW[j][c] = sum_p part[p][c][j] + part[p][64 + c][j];   dR[c][j] = sum_p part[p][32 + c][j] + part[p][96 + c][j]
// block 64 (when part_b is given): dr[c] = sum_p part_b[p][c], the same two-level fixed order
__global__ void __launch_bounds__(256) k_bwd_tc_reduce(const float* __restrict__ part, int P, float* __restrict__ dw,
                                                       float* __restrict__ d_res_w, const float* __restrict__ part_b,
                                                       int Pb, float* __restrict__ d_res_b) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (blockIdx.x == 64) {
    const int per = (Pb + 7) / 8, p0 = warp * per, p1 = min(Pb, p0 + per);
    float sb = 0.f;
    for (int p = p0; p < p1; ++p) sb += part_b[(int64_t)p * 32 + lane];
    red[warp][lane] = sb;
    __syncthreads();
    if (warp == 0) {
      float t = red[0][lane];
#pragma unroll
      for (int w = 1; w < 8; ++w) t += red[w][lane];
      d_res_b[lane] = t;
    }
    return;
  }
  const int o = blockIdx.x * 32 + lane;          // 0..2047
  const int which = o >> 10, a0 = (o >> 5) & 31, b0 = o & 31;
  // dW[j = a0][c = b0]: rows c, 64 + c, column j;  dR[c = a0][j = b0]: rows 32 + c, 96 + c, column j
  const int row = which == 0 ? b0 : 32 + a0, col = which == 0 ? a0 : b0;
  const int per = (P + 7) / 8, p0 = warp * per, p1 = min(P, p0 + per);
  float s_main = 0.f, s_corr = 0.f;
  for (int p = p0; p < p1; ++p) {
    s_main += part[((int64_t)p * 128 + row) * 32 + col];
    s_corr += part[((int64_t)p * 128 + row + 64) * 32 + col];
  }
  red[warp][lane] = s_main + s_corr;
  __syncthreads();
  if (warp == 0) {
    float s = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) s += red[w][lane];
    (which == 0 ? dw : d_res_w)[a0 * 32 + b0] = s;
  }
}

int launch_bwd_tc_reduce(const float* part, int P, float* dw, float* d_res_w, const float* part_b, int Pb,
                         float* d_res_b, void* stream) {
  MGCN_LAUNCH(k_bwd_tc_reduce, part_b ? 65 : 64, 256, 0, stream, part, P, dw, d_res_w, part_b, Pb, d_res_b);
  return MGCN_OK;
}

int bwd_tc_grid(int64_t N) {
  const int64_t tiles = ceil_div(N > 0 ? N : 1, kTRows);
  return (int)(tiles < kNumSMs ? tiles : kNumSMs);
}

size_t bwd_tc_workspace_floats(int64_t N) { return (size_t)bwd_tc_grid(N) * (128 * 32 + 32); }
size_t bwd_tc_bias_workspace_floats(int64_t N) { return mask_bits_colsum_workspace_floats(N); }

int launch_layer_bwd_tc(const float* dxw, const float* gy, const float* x, const float* x_scale, const float* w, const float* res_w,
                        const uint32_t* hmask_prev, const float* post, int64_t N, float* gy_prev, float* gs_prev,
                        float* dw, float* d_res_w, float* d_res_b, float* ws, void* stream,
                        const uint32_t* hmask_cur, float bias_scale, float* d_bias) {
  const int P = bwd_tc_grid(N);
  BwdTcArgs a{};
  a.dxw = dxw; a.gy = gy; a.x = x; a.x_scale = x_scale; a.w = w; a.res_w = res_w; a.hmask_prev = hmask_prev; a.post = post;
  a.gy_prev = gy_prev; a.gs_prev = gs_prev;
  a.part_t = ws;
  a.part_b = ws + (size_t)P * 128 * 32;
  a.n_rows = N;
  // the attribute belongs to (function, device): set on every call (cheap), so a second GPU in the same process
  // gets it too and a failure is reported every time
  cudaError_t attr_err = cudaSuccess;
  {
    attr_err = cudaFuncSetAttribute(k_layer_bwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, kBwdTcSmem);
  }
  MGCN_CHECK_CUDA(attr_err);
  MGCN_LAUNCH(k_layer_bwd_tc, P, kBwdTcThreads, kBwdTcSmem, stream, a);
  const int rc = launch_bwd_tc_reduce(a.part_t, P, dw, d_res_w, a.part_b, P, d_res_b, stream);   // dW, dR and dr: one launch
  if (rc != MGCN_OK || !d_bias) return rc;
  // the node-model bias gradient as its own pass over gy: summed by the producer warps above, next to dr, the kernel
  // needs 8 more live registers than its 80 and spills (profiles/bias_ptxas.log)
  return launch_mask_bits_colsum(gy, hmask_cur, bias_scale, N, d_bias, ws + bwd_tc_workspace_floats(N), stream);
}

// ---- masked column sum: the node-model bias gradient,  d_bias[c] = scale * sum_i bit c of bits[i] * gy[i][c] ----
// Lane 8 q + k of a warp reads columns 4k .. 4k + 3 of row 4 w + q of the block's 32-row step: one float4 per lane, 512
// contiguous bytes per warp.  The 4 rows of a warp are added by a fixed butterfly, the 8 warps of a block in order,
// the per-block partials by one block (8 contiguous runs, then the runs in order).  The grid depends on N (and the
// SM count) only, so the result is the same from run to run.
constexpr int kColsumRows = 32;   // rows per block and step: 8 warps x 4 rows
__global__ void __launch_bounds__(256) k_mask_bits_colsum(const float* __restrict__ gy, const uint32_t* __restrict__ bits,
                                                          int64_t n_rows, float* __restrict__ part) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane >> 3, k = lane & 7;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  const int64_t stride = (int64_t)gridDim.x * kColsumRows;
  const uint64_t pol = policy_evict_first();
#pragma unroll 4
  for (int64_t r = (int64_t)blockIdx.x * kColsumRows + 4 * warp + q; r < n_rows; r += stride) {
    const float4 g = ld_f4_hint(gy + r * kTH + 4 * k, pol);
    const uint32_t m = __ldg(bits + r) >> (4 * k);
    acc[0] += (m & 1u) ? g.x : 0.f;
    acc[1] += (m & 2u) ? g.y : 0.f;
    acc[2] += (m & 4u) ? g.z : 0.f;
    acc[3] += (m & 8u) ? g.w : 0.f;
  }
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    float v = acc[t];
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    if (q == 0) red[warp][4 * k + t] = v;
  }
  __syncthreads();
  if (warp == 0) {
    float s = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) s += red[w][lane];
    part[(int64_t)blockIdx.x * 32 + lane] = s;
  }
}

// out[c] = scale * sum_p part[p][c]: warp w sums a contiguous run of partials, warp 0 adds the 8 runs in order
__global__ void __launch_bounds__(256) k_colsum_reduce(const float* __restrict__ part, int P, float scale,
                                                       float* __restrict__ out) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int per = (P + 7) / 8, p0 = warp * per, p1 = min(P, p0 + per);
  float s = 0.f;
  for (int p = p0; p < p1; ++p) s += part[(int64_t)p * 32 + lane];
  red[warp][lane] = s;
  __syncthreads();
  if (warp == 0) {
    float t = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) t += red[w][lane];
    out[lane] = t * scale;
  }
}

static int colsum_grid(int64_t N) {
  const int64_t blocks = ceil_div(N > 0 ? N : 1, kColsumRows);
  return (int)(blocks < (int64_t)kNumSMs * 8 ? blocks : (int64_t)kNumSMs * 8);
}

size_t mask_bits_colsum_workspace_floats(int64_t N) { return (size_t)colsum_grid(N) * 32; }

int launch_mask_bits_colsum(const float* gy, const uint32_t* bits, float scale, int64_t N, float* d_bias, float* ws,
                            void* stream) {
  const int P = colsum_grid(N);
  MGCN_LAUNCH(k_mask_bits_colsum, P, 256, 0, stream, gy, bits, N, ws);
  MGCN_LAUNCH(k_colsum_reduce, 1, 256, 0, stream, ws, P, scale, d_bias);
  return MGCN_OK;
}

}  // namespace mgcn
