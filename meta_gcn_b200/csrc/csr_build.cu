// edge_index (int64 COO) -> row-owned int32 structure: stable LSD radix sort + segment offsets.
//
// Ordering contract (SURVEY.md §8 a12): inside a row, entries keep their edge_index order, which is
// the order the reference's CPU scatter_add (common.py:56-59 -> torch_scatter 1.x ->
// Tensor.scatter_add_) accumulates them in.  Everything here is integer work: results are
// bit-exact and independent of scheduling (integer atomics only feed commutative counts).
#include "common.cuh"

namespace mgcn {

// ------------------------------------------------------------------------------------------------
// exclusive scan (int32), reduce-then-scan, in-place safe
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 1024;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ int32_t warp_inclusive_scan(int32_t v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int32_t o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += o;
  }
  return v;
}

// exclusive scan of one value per thread across a 1024-thread block; returns block total via *total
__device__ __forceinline__ int32_t block_exclusive_scan(int32_t v, int32_t* total) {
  __shared__ int32_t warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t inc = warp_inclusive_scan(v, lane);
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int32_t ws = warp_sums[lane];
    int32_t winc = warp_inclusive_scan(ws, lane);
    warp_sums[lane] = winc - ws;  // exclusive
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  int32_t res = warp_sums[warp] + inc - v;
  __syncthreads();  // warp_sums reusable by the caller's next call
  return res;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_tile_sums(const int32_t* __restrict__ in,
                                                                 int64_t n,
                                                                 int32_t* __restrict__ tile_sums) {
  __shared__ int32_t total;
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  int32_t s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) s += in[base + i];
  (void)block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// single block: exclusive scan of tile_sums[0..nt) in place
__global__ void __launch_bounds__(kScanThreads) k_scan_tile_offsets(int32_t* tile_sums, int nt) {
  __shared__ int32_t total;
  int32_t carry = 0;
  for (int base = 0; base < nt; base += kScanThreads) {
    const int i = base + threadIdx.x;
    const int32_t v = i < nt ? tile_sums[i] : 0;
    const int32_t ex = block_exclusive_scan(v, &total);
    if (i < nt) tile_sums[i] = carry + ex;
    carry += total;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kScanThreads) k_scan_apply(const int32_t* in, int32_t* out,
                                                             int64_t n,
                                                             const int32_t* __restrict__ tile_off) {
  __shared__ int32_t total;
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  int32_t v[kScanItems];
  int32_t s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = base + i < n ? in[base + i] : 0;
    s += v[i];
  }
  int32_t run = tile_off[blockIdx.x] + block_exclusive_scan(s, &total);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = run;
    run += v[i];
  }
}

// short inputs (the structures of small-graph batches: a few thousand rows): ONE block walks the tiles with a running
// carry — one launch instead of three; integer sums, same result
__global__ void __launch_bounds__(kScanThreads) k_scan_small(const int32_t* in, int32_t* out, int64_t n) {
  __shared__ int32_t total;
  int32_t carry = 0;
  for (int64_t tile0 = 0; tile0 < n; tile0 += kScanTile) {
    const int64_t base = tile0 + (int64_t)threadIdx.x * kScanItems;
    int32_t v[kScanItems];
    int32_t s = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
      v[i] = base + i < n ? in[base + i] : 0;
      s += v[i];
    }
    int32_t run = carry + block_exclusive_scan(s, &total);
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
      if (base + i < n) out[base + i] = run;
      run += v[i];
    }
    carry += total;
    __syncthreads();
  }
}
constexpr int64_t kScanSmallMax = 1 << 16;

static size_t scan_tiles(int64_t n) { return (size_t)ceil_div(n > 0 ? n : 1, kScanTile); }

// tile_sums must hold scan_tiles(n) ints
static int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, int32_t* tile_sums,
                              void* stream) {
  if (n <= 0) return MGCN_OK;
  if (n <= kScanSmallMax) {
    MGCN_LAUNCH(k_scan_small, 1, kScanThreads, 0, stream, in, out, n);
    return MGCN_OK;
  }
  const int nt = (int)scan_tiles(n);
  MGCN_LAUNCH(k_scan_tile_sums, nt, kScanThreads, 0, stream, in, n, tile_sums);
  MGCN_LAUNCH(k_scan_tile_offsets, 1, kScanThreads, 0, stream, tile_sums, nt);
  MGCN_LAUNCH(k_scan_apply, nt, kScanThreads, 0, stream, in, out, n, tile_sums);
  return MGCN_OK;
}

// ------------------------------------------------------------------------------------------------
// keys + row histogram
// ------------------------------------------------------------------------------------------------
template <typename IndexT>   // int64_t (the reference's edge_index dtype) or int32_t (half the H2D bytes)
__global__ void __launch_bounds__(256) k_make_keys(const IndexT* __restrict__ ei, int64_t E,
                                                   int64_t N, int by, int loop_mode,
                                                   int64_t total, uint32_t* __restrict__ keys,
                                                   int32_t* __restrict__ counts,
                                                   int32_t* __restrict__ bad_index) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  // warp-uniform loop bound: every lane reaches the match below in every iteration
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x - lane); base < total; base += stride) {
    const int64_t e = base + lane;
    const bool in = e < total;
    uint32_t key = 0xffffffffu;
    if (in) {
      if (e < E) {
        const int64_t s = (int64_t)ei[e], d = (int64_t)ei[E + e];
        const bool ok = s >= 0 && s < N && d >= 0 && d < N;
        if (!ok) {
          *bad_index = 1;
          key = (uint32_t)N;
        } else if (loop_mode != 0 && s == d) {
          key = (uint32_t)N;  // dropped
        } else {
          key = (uint32_t)(by == 0 ? s : d);
        }
      } else {
        key = (uint32_t)(e - E);  // appended self loop of node e-E (loop_mode 2)
      }
      if (keys != nullptr) keys[e] = key;   // a sort-free build needs no keys
    }
    // row histogram: the lanes of a warp that hold the same key add once (an ordered list has ~10 equal keys in a
    // row: a tenth of the atomics; integer sums, so the grouping does not change the result)
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (in && key < (uint32_t)N && lane == __ffs(peers) - 1) atomicAdd(&counts[key], __popc(peers));
  }
}

// ------------------------------------------------------------------------------------------------
// stable LSD radix sort of (key, position) pairs, 8-bit digits.
// Tile = 8 warps x 16 rounds x 32 lanes; a warp owns 512 consecutive items, so the stable order
// inside a tile is (warp, round, lane).
// ------------------------------------------------------------------------------------------------
constexpr int kRsWarps = 8;
constexpr int kRsRounds = 16;
constexpr int kRsTile = kRsWarps * 32 * kRsRounds;

__global__ void __launch_bounds__(256) k_radix_hist(const uint32_t* __restrict__ keys, int64_t n,
                                                    int shift, int32_t* __restrict__ block_hist,
                                                    int num_blocks) {
  __shared__ int32_t wh[kRsWarps][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kRsWarps * 256; i += 256) (&wh[0][0])[i] = 0;
  __syncthreads();
  const int64_t wbase = (int64_t)blockIdx.x * kRsTile + (int64_t)warp * (32 * kRsRounds);
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll 4
  for (int r = 0; r < kRsRounds; ++r) {
    const int64_t idx = wbase + r * 32 + lane;
    const uint32_t d = idx < n ? ((keys[idx] >> shift) & 255u) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (d < 256u && (peers & lt) == 0u) wh[warp][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  int32_t s = 0;
#pragma unroll
  for (int w = 0; w < kRsWarps; ++w) s += wh[w][threadIdx.x];
  block_hist[(int64_t)threadIdx.x * num_blocks + blockIdx.x] = s;
}

// Scatter pass.  The tile is first ordered by digit in shared memory (stable: digit, then warp, round, lane)
// and then written out run by run, so the items of one digit leave as one contiguous, coalesced run per
// array (measured at 37.5 M pairs: 0.70 ms with direct 4-byte scatters from registers, each its own sector).
__global__ void __launch_bounds__(256)
    k_radix_scatter(const uint32_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in,
                    uint32_t* __restrict__ keys_out, int32_t* __restrict__ vals_out, int64_t n,
                    int shift, const int32_t* __restrict__ block_off, int num_blocks) {
  __shared__ int32_t wh[kRsWarps][256];     // per-warp digit counts, then tile-local start of (digit, warp)
  __shared__ int32_t dig_start[256];        // tile-local start of the digit's run
  __shared__ int32_t dig_gbase[256];        // global position of the run's first item
  __shared__ int32_t scan_w[8];
  __shared__ uint32_t s_key[kRsTile];
  __shared__ int32_t s_val[kRsTile];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kRsWarps * 256; i += 256) (&wh[0][0])[i] = 0;
  __syncthreads();
  const int64_t tbase = (int64_t)blockIdx.x * kRsTile;
  const int64_t wbase = tbase + (int64_t)warp * (32 * kRsRounds);
  const unsigned lt = (1u << lane) - 1u;
  uint32_t key[kRsRounds];
#pragma unroll
  for (int r = 0; r < kRsRounds; ++r) {
    const int64_t idx = wbase + r * 32 + lane;
    key[r] = idx < n ? keys_in[idx] : 0u;
    const uint32_t d = idx < n ? ((key[r] >> shift) & 255u) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (d < 256u && (peers & lt) == 0u) wh[warp][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  {
    // thread d: total of digit d in the tile -> exclusive scan over the 256 digits -> starts per (digit, warp)
    const int d = threadIdx.x;
    int32_t tot = 0;
#pragma unroll
    for (int w = 0; w < kRsWarps; ++w) tot += wh[w][d];
    int32_t inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) scan_w[warp] = inc;
    __syncthreads();
    int32_t wpre = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) wpre += (w < warp) ? scan_w[w] : 0;
    int32_t start = wpre + inc - tot;
    dig_start[d] = start;
    dig_gbase[d] = block_off[(int64_t)d * num_blocks + blockIdx.x];
#pragma unroll
    for (int w = 0; w < kRsWarps; ++w) {
      const int32_t c = wh[w][d];
      wh[w][d] = start;
      start += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kRsRounds; ++r) {
    const int64_t idx = wbase + r * 32 + lane;
    const bool valid = idx < n;
    const uint32_t d = valid ? ((key[r] >> shift) & 255u) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & lt);
    int32_t lp = 0;
    if (valid) lp = wh[warp][d] + rank;
    __syncwarp();
    if (valid && rank == 0) wh[warp][d] += __popc(peers);
    __syncwarp();
    if (valid) {
      s_key[lp] = key[r];
      s_val[lp] = vals_in ? vals_in[idx] : (int32_t)idx;
    }
  }
  __syncthreads();
  const int64_t rem = n - tbase;
  const int cnt = rem < kRsTile ? (int)rem : kRsTile;
  for (int k = threadIdx.x; k < cnt; k += 256) {
    const uint32_t kk = s_key[k];
    const uint32_t d = (kk >> shift) & 255u;
    const int32_t dst = dig_gbase[d] + (k - dig_start[d]);
    keys_out[dst] = kk;
    vals_out[dst] = s_val[k];
  }
}

template <typename IndexT>
__global__ void __launch_bounds__(256)
    k_finalize(const IndexT* __restrict__ ei, int64_t E, int by, int64_t total,
               const int32_t* __restrict__ sorted_pos, const int32_t* __restrict__ rowptr,
               int64_t N, int32_t* __restrict__ nbr, int32_t* __restrict__ perm) {
  const int32_t kept = rowptr[N];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride) {
    if (k < kept) {
      const int32_t p = sorted_pos[k];
      perm[k] = p;
      nbr[k] = p < E ? (int32_t)(by == 0 ? ei[E + p] : ei[p]) : (int32_t)(p - E);
    } else {
      perm[k] = -1;
      nbr[k] = 0;
    }
  }
}

// Hub rows (longer than `threshold`) are cut into segments of `threshold` entries.  The order in
// which hubs claim table slots is arbitrary (atomic counters) but never reaches the results: each
// hub's segments are contiguous and combined in segment order.
__global__ void __launch_bounds__(256)
    k_find_hubs(const int32_t* __restrict__ rowptr, int64_t N, int32_t threshold,
                int32_t* __restrict__ hub_rows, int32_t* __restrict__ hub_seg0, int64_t hub_cap,
                int32_t* __restrict__ hub_count, int32_t* __restrict__ seg_row,
                int32_t* __restrict__ seg_beg, int64_t seg_cap, int32_t* __restrict__ seg_count) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int32_t beg = rowptr[i];
  const int32_t len = rowptr[i + 1] - beg;
  if (len > threshold) {
    const int32_t nseg = (len + threshold - 1) / threshold;
    const int32_t k = atomicAdd(hub_count, 1);
    const int32_t s0 = atomicAdd(seg_count, nseg);
    if (k < hub_cap && (int64_t)s0 + nseg <= seg_cap) {
      hub_rows[k] = (int32_t)i;
      hub_seg0[k] = s0;
      for (int32_t q = 0; q < nseg; ++q) {
        seg_row[s0 + q] = (int32_t)i;
        seg_beg[s0 + q] = beg + q * threshold;
      }
    }
  }
}

// work-order key: (locality window, row length clipped to 1023)
constexpr int kOrderWindowShift = 14;  // 16384 rows: 2 MB of H=32 features stay L2/L1-local
constexpr int kOrderLenBits = 10;

__global__ void __launch_bounds__(256) k_order_keys(const int32_t* __restrict__ rowptr, int64_t N,
                                                    uint32_t* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int32_t len = rowptr[i + 1] - rowptr[i];
  if (len > (1 << kOrderLenBits) - 1) len = (1 << kOrderLenBits) - 1;
  keys[i] = ((uint32_t)(i >> kOrderWindowShift) << kOrderLenBits) | (uint32_t)len;
}

// Work descriptors {row, beg, end, partial_slot} in work order (see mgcn_csr_t::tasks) and the index
// stream permuted into the same order (nbr_w).  A task is a row within the hub threshold or one
// segment of a hub row; task ids: [0,N) = rows, [N, N+seg_cap) = segment slots.  Work order = stable
// sort by (16384-row locality window, length; segments behind the rows of their window), so a hub's
// segments run while its window's features are L2-resident (measured: with all segments queued
// behind the last row, their 15 % of the gathers missed L2 and doubled the DRAM reads).
// Steps: keys -> radix sort -> entry count per task -> exclusive scan (task p starts where task
// p-1 ends) -> descriptors + copy of the entries.
__global__ void __launch_bounds__(256)
    k_task_keys(const int32_t* __restrict__ rowptr, int64_t N, const int32_t* __restrict__ seg_row,
                const int32_t* __restrict__ seg_count, int64_t seg_cap, uint32_t* __restrict__ keys) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= N + seg_cap) return;
  constexpr uint32_t kSegLen = 1u << kOrderLenBits;  // sorts behind every row length
  uint32_t key;
  if (s < N) {
    int32_t len = rowptr[s + 1] - rowptr[s];
    if (len > (int32_t)kSegLen - 1) len = kSegLen - 1;
    key = ((uint32_t)(s >> kOrderWindowShift) << (kOrderLenBits + 1)) | (uint32_t)len;
  } else {
    int64_t ns = *seg_count;
    if (ns > seg_cap) ns = seg_cap;
    const int64_t q = s - N;
    if (q < ns) {
      key = ((uint32_t)(seg_row[q] >> kOrderWindowShift) << (kOrderLenBits + 1)) | kSegLen;
    } else {
      key = ((uint32_t)(((N > 0 ? N - 1 : 0) >> kOrderWindowShift) + 1) << (kOrderLenBits + 1));  // padding: last
    }
  }
  keys[s] = key;
}

// entry count of the task at work position p; entry n_tasks is a zero terminator (scan -> total)
__global__ void __launch_bounds__(256)
    k_task_lengths(const int32_t* __restrict__ tid, const int32_t* __restrict__ rowptr, int64_t N,
                   const int32_t* __restrict__ seg_row, const int32_t* __restrict__ seg_beg,
                   const int32_t* __restrict__ seg_count, int64_t seg_cap, int32_t threshold,
                   int32_t* __restrict__ len_w) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_tasks = N + seg_cap;
  if (p > n_tasks) return;
  int32_t len = 0;
  if (p < n_tasks) {
    const int64_t s = tid[p];
    if (s < N) {
      len = rowptr[s + 1] - rowptr[s];
      if (len > threshold) len = 0;  // hub row: covered by its segments
    } else {
      int64_t ns = *seg_count;
      if (ns > seg_cap) ns = seg_cap;
      const int64_t q = s - N;
      if (q < ns) len = min(threshold, rowptr[seg_row[q] + 1] - seg_beg[q]);
    }
  }
  len_w[p] = len;
}

// one 8-lane group per work position: descriptor + copy of the task's entries into work order
__global__ void __launch_bounds__(256)
    k_make_tasks(const int32_t* __restrict__ tid, const int32_t* __restrict__ rowptr, int64_t N,
                 const int32_t* __restrict__ seg_row, const int32_t* __restrict__ seg_beg,
                 const int32_t* __restrict__ seg_count, int64_t seg_cap, int32_t threshold,
                 const int32_t* __restrict__ wpos, const int32_t* __restrict__ nbr,
                 int4* __restrict__ tasks, int32_t* __restrict__ nbr_w) {
  const int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int sub = threadIdx.x & 7;
  if (p >= N + seg_cap) return;
  const int32_t w0 = wpos[p], w1 = wpos[p + 1];
  const int64_t s = tid[p];
  int32_t row = -1, src = 0, slot = 0;
  if (s < N) {
    src = rowptr[s];
    if (rowptr[s + 1] - src <= threshold) row = (int32_t)s;
  } else {
    int64_t ns = *seg_count;
    if (ns > seg_cap) ns = seg_cap;
    const int64_t q = s - N;
    if (q < ns) {
      row = seg_row[q];
      src = seg_beg[q];
      slot = (int32_t)q + 1;
    }
  }
  if (sub == 0) tasks[p] = make_int4(row, w0, w1, slot);
  for (int32_t k = w0 + sub; k < w1; k += 8) nbr_w[k] = nbr[src + (k - w0)];
}

__global__ void __launch_bounds__(256) k_copy_i32(const int32_t* __restrict__ in, int64_t n,
                                                  int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}

__global__ void __launch_bounds__(256) k_degree(const int32_t* __restrict__ rowptr, int64_t N,
                                                float* __restrict__ deg) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) deg[i] = (float)(rowptr[i + 1] - rowptr[i]);
}

// one thread per row, sequential in row order: deterministic and equal to the reference's
// edge-order scatter_add of weights (gcn_base_models.py:126)
__global__ void __launch_bounds__(256)
    k_weighted_degree(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                      const float* __restrict__ ew, int64_t E, float loop_w, int64_t N,
                      float* __restrict__ deg) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float s = 0.f;
  for (int32_t k = rowptr[i]; k < rowptr[i + 1]; ++k) {
    const int32_t p = perm[k];
    s = __fadd_rn(s, p < E ? ew[p] : loop_w);
  }
  deg[i] = s;
}

__global__ void __launch_bounds__(256) k_gcn_norm(const float* __restrict__ deg, int64_t N, int mode,
                                                  float* __restrict__ dis) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float d = deg[i];
  // deg.pow(-0.5) / deg.pow(-1) on the CPU reference are 1/sqrt(d) and 1/d, both correctly rounded
  float v = mode == 0 ? __fdiv_rn(1.0f, __fsqrt_rn(d)) : __fdiv_rn(1.0f, d);
  if (v == __int_as_float(0x7f800000)) v = 0.f;  // gcn_base_models.py:135 (only +inf is masked)
  dis[i] = v;
}

__global__ void __launch_bounds__(256)
    k_permute_vals(const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr, int64_t N,
                   int64_t total, const float* __restrict__ vin, int64_t E, float loop_value,
                   float* __restrict__ vout) {
  const int32_t kept = rowptr[N];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride) {
    float v = 0.f;
    if (k < kept) {
      const int32_t p = perm[k];
      v = p < E ? vin[p] : loop_value;
    }
    vout[k] = v;
  }
}

static int grid_for(int64_t n, int block, int max_blocks = kNumSMs * 32) {
  int64_t g = ceil_div(n > 0 ? n : 1, block);
  if (g > max_blocks) g = max_blocks;
  return (int)g;
}

static int radix_passes_for(uint64_t max_key) {
  int bits = 1;
  while ((uint64_t(1) << bits) <= max_key) ++bits;
  return (bits + 7) / 8;
}

// stable sort of (keys, position) by key; keys_a holds the input keys, initial values are the
// positions 0..n-1.  *sorted_vals points at the buffer holding the sorted positions.
static int radix_sort_positions(uint32_t* keys_a, uint32_t* keys_b, int32_t* vals_a, int32_t* vals_b,
                                int64_t n, uint64_t max_key, int32_t* block_hist,
                                int32_t* tile_sums, const int32_t** sorted_vals, void* stream,
                                const int32_t* vals_init = nullptr) {
  const int num_blocks = (int)ceil_div(n > 0 ? n : 1, kRsTile);
  const int64_t hist_len = (int64_t)256 * num_blocks;
  const int passes = radix_passes_for(max_key);
  const uint32_t* kin = keys_a;
  uint32_t* kout = keys_b;
  const int32_t* vin = vals_init;  // nullptr: identity on the first pass
  int32_t* vout = (vals_init == vals_a) ? vals_b : vals_a;
  for (int p = 0; p < passes; ++p) {
    const int shift = 8 * p;
    MGCN_LAUNCH(k_radix_hist, num_blocks, 256, 0, stream, kin, n, shift, block_hist, num_blocks);
    int rc = exclusive_scan_i32(block_hist, block_hist, hist_len, tile_sums, stream);
    if (rc != MGCN_OK) return rc;
    MGCN_LAUNCH(k_radix_scatter, num_blocks, 256, 0, stream, kin, vin, kout, vout, n, shift,
                block_hist, num_blocks);
    uint32_t* old_in = const_cast<uint32_t*>(kin);
    kin = kout;
    kout = old_in;
    vin = vout;
    vout = (vout == vals_a) ? vals_b : vals_a;
  }
  *sorted_vals = vin;
  return MGCN_OK;
}

// ------------------------------------------------------------------------------------------------
// Edge preprocessing that DEFINES the botnet edge order (data_procs/undirected.py:6-35: both directions,
// sort-unique by row*N+col keeping the first occurrence; loop.py:13-17: (i,i) for every node appended at
// the END; data_add_degree.py:45-65: out-degree incl. the loop as float32).  Lexicographic (row, col)
// order = stable sort by col, then stable sort by row, with the same radix machinery as the structure
// build; duplicates are adjacent afterwards.  Element i of the (virtually) doubled list is
// (r[i], c[i]) for i < E and (c[i-E], r[i-E]) for i >= E.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t pre_endpoint(const int64_t* __restrict__ ei, int64_t E, int64_t i, int which) {
  // which: 0 = row (source), 1 = col (target) of doubled element i
  const bool flip = i >= E;
  const int64_t e = flip ? i - E : i;
  return (which == 0) != flip ? ei[e] : ei[E + e];
}

__global__ void __launch_bounds__(256)
    k_pre_keys(const int64_t* __restrict__ ei, int64_t E, int64_t M, int64_t N, int which,
               const int32_t* __restrict__ pos, uint32_t* __restrict__ keys, int32_t* __restrict__ bad) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < M; k += stride) {
    const int64_t i = pos ? pos[k] : k;
    int64_t v = pre_endpoint(ei, E, i, which);
    if (v < 0 || v >= N) {
      *bad = 1;
      v = 0;
    }
    keys[k] = (uint32_t)v;
  }
}

__global__ void __launch_bounds__(256)
    k_pre_flags(const int64_t* __restrict__ ei, int64_t E, int64_t M, const int32_t* __restrict__ pos,
                int32_t* __restrict__ flags) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k <= M; k += stride) {
    int32_t f = 0;
    if (k < M) {
      f = 1;
      if (k > 0) {
        const int64_t a = pos[k], b = pos[k - 1];
        if (pre_endpoint(ei, E, a, 0) == pre_endpoint(ei, E, b, 0) &&
            pre_endpoint(ei, E, a, 1) == pre_endpoint(ei, E, b, 1))
          f = 0;
      }
    }
    flags[k] = f;  // entry M is a zero terminator: the scan yields the number of unique edges
  }
}

__global__ void __launch_bounds__(256)
    k_pre_compact(const int64_t* __restrict__ ei, int64_t E, int64_t M, const int32_t* __restrict__ pos,
                  const int32_t* __restrict__ flags, const int32_t* __restrict__ idx, int64_t cap,
                  int64_t N, int64_t* __restrict__ out, int32_t* __restrict__ perm,
                  int32_t* __restrict__ degi) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < M; k += stride) {
    if (!flags[k]) continue;
    const int64_t i = pos[k];
    const int64_t r = pre_endpoint(ei, E, i, 0), c = pre_endpoint(ei, E, i, 1);
    const int32_t o = idx[k];
    out[o] = r;
    out[cap + o] = c;
    perm[o] = (int32_t)i;
    if (r >= 0 && r < N) atomicAdd(degi + r, 1);   // integer count: order-independent (bad ids are flagged)
  }
}

__global__ void __launch_bounds__(256)
    k_pre_finish(const int32_t* __restrict__ idx, int64_t M, int64_t N, int add_loops, int64_t cap,
                 int64_t* __restrict__ out, int32_t* __restrict__ perm, const int32_t* __restrict__ degi,
                 float* __restrict__ deg, int64_t* __restrict__ count) {
  const int64_t unique = idx[M];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    if (add_loops) {
      out[unique + i] = i;
      out[cap + unique + i] = i;
      perm[unique + i] = -1;
    }
    deg[i] = (float)(degi[i] + (add_loops ? 1 : 0));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *count = unique + (add_loops ? N : 0);
}

}  // namespace mgcn

using namespace mgcn;

extern "C" int mgcn_csr_capacities(int64_t E, int64_t N, int loop_mode, int32_t hub_threshold,
                                   int64_t* nnz_cap, int64_t* hub_cap, int64_t* seg_cap) {
  MGCN_REQUIRE(nnz_cap && hub_cap && seg_cap, MGCN_ERR_NULL);
  MGCN_REQUIRE(E >= 0 && N >= 0 && hub_threshold >= 1, MGCN_ERR_RANGE);
  MGCN_REQUIRE(loop_mode >= 0 && loop_mode <= 2, MGCN_ERR_SHAPE);
  const int64_t total = E + (loop_mode == 2 ? N : 0);
  *nnz_cap = total;
  *hub_cap = total / hub_threshold + 1;              // every hub owns > hub_threshold entries
  *seg_cap = total / hub_threshold + *hub_cap + 1;   // sum ceil(len/T) <= nnz/T + hubs
  return MGCN_OK;
}

// Entries of a list that is ALREADY in (source, target) lexicographic order — optionally followed by the N self loops
// (0,0) .. (N-1,N-1), the layout data_procs/undirected.py:6-35 + loop.py:13-17 give every botnet graph — need no
// sort: the stable grouping by source is "prefix entry e of source s -> e (+ s loops of smaller rows), loop i -> end
// of row i".  For a symmetric list the grouping by target is the same row contents (sources ascending, loop last),
// and the edge that sits at a by-target position is the mirror (d, s) of the by-source one, found by a binary search
// in row d.  `dups` != 0: the list may repeat an entry; the k-th copy of (s, d) is paired with the k-th copy of (d, s).
// graph of list position e in a batch: edge_off[g] <= e < edge_off[g+1]  (G <= a few hundred: a short binary search)
__device__ __forceinline__ int segment_of(const int32_t* __restrict__ off, int G, int64_t v) {
  int lo = 0, hi = G;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((int64_t)off[mid] <= v) lo = mid; else hi = mid;
  }
  return lo;
}
// the same with the previous answer as a hint: a thread's entries advance monotonically and a graph of a batch spans
// millions of them, so two cached loads usually replace the dependent chain of the search
__device__ __forceinline__ int segment_of_hint(const int32_t* __restrict__ off, int G, int64_t v, int hint) {
  if (hint >= 0 && hint < G && (int64_t)off[hint] <= v && v < (int64_t)off[hint + 1]) return hint;
  return segment_of(off, G, v);
}

// A BATCH of such lists (Batch.from_data_list: graph after graph, node ids shifted; dataloader.py:11) is the same
// layout per graph: node_off / edge_off [G+1] delimit the graphs (G = 0: the whole list is one graph).
template <typename IndexT>
__global__ void __launch_bounds__(256)
    k_fill_presorted(const IndexT* __restrict__ ei, int64_t E, int64_t N, int by, int tail, int dups, int G,
                     const int32_t* __restrict__ node_off, const int32_t* __restrict__ edge_off,
                     const int32_t* __restrict__ rowptr, int32_t* __restrict__ nbr, int32_t* __restrict__ perm) {
  int seg_hint = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    int64_t n0 = 0, e0 = 0, ng = N, eg = E;   // this entry's graph: first node, first entry, sizes
    if (G > 0) {
      const int g = seg_hint = segment_of_hint(edge_off, G, e, seg_hint);
      n0 = node_off[g];
      e0 = edge_off[g];
      ng = node_off[g + 1] - n0;
      eg = edge_off[g + 1] - e0;
    }
    const int64_t Ep = e0 + (tail ? eg - ng : eg);   // end of the graph's sorted prefix
    if (e >= Ep) {
      const int64_t i = n0 + (e - Ep);
      const int32_t k = rowptr[i + 1] - 1;
      nbr[k] = (int32_t)i;
      perm[k] = (int32_t)e;
      continue;
    }
    const int64_t s = (int64_t)ei[e], d = (int64_t)ei[E + e];
    if (s < 0 || s >= N || d < 0 || d >= N) continue;   // flagged by k_make_keys
    if (by == 0) {
      const int64_t k = e + (tail ? s - n0 : 0);
      nbr[k] = (int32_t)d;
      perm[k] = (int32_t)e;
      continue;
    }
    // first position of value v among the targets of prefix row r
    auto lower = [&](int64_t r, int64_t v) {
      int64_t lo = rowptr[r] - (tail ? r : 0), hi = rowptr[r + 1] - (tail ? r + 1 : 0);
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)ei[E + mid] < v) lo = mid + 1; else hi = mid;
      }
      return lo;
    };
    const int64_t off = dups ? e - lower(s, d) : 0;
    const int64_t k = lower(d, s) + off + (tail ? d : 0);
    nbr[k] = (int32_t)s;
    perm[k] = (int32_t)e;
  }
}

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
// out[0..3]: the multiset fingerprints (as k_edge_fingerprint; accumulated here in the same pass over the list — one
// read of edge_index instead of two); out[4] entries e with (src,dst)[e] > (src,dst)[e+1]
// over the whole list, out[5] the same over the first E-N entries, out[6] entries of the last N that are not the
// loop (e-(E-N), e-(E-N)), out[7] adjacent equal entries (whole list).  An entry with an endpoint outside [0, N) (in a
// batch: outside its graph's node range) counts once more in out[4] and out[5].
template <typename IndexT>
__global__ void __launch_bounds__(256) k_edge_order_check(const IndexT* __restrict__ ei, int64_t E, int64_t N, int G,
                                                          const int32_t* __restrict__ node_off,
                                                          const int32_t* __restrict__ edge_off,
                                                          unsigned long long* __restrict__ out) {
  unsigned long long f[4] = {0ull, 0ull, 0ull, 0ull}, h[4] = {0ull, 0ull, 0ull, 0ull};
  int seg_hint = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t s = (int64_t)ei[e], d = (int64_t)ei[E + e];
    {
      const uint64_t a = (uint64_t)s, b = (uint64_t)d;
      const uint64_t ab = a * 0x9e3779b97f4a7c15ull + b, ba = b * 0x9e3779b97f4a7c15ull + a;
      h[0] += mix64(ab);
      h[1] += mix64(ba);
      h[2] += mix64(ab ^ 0xd6e8feb86659fd93ull);
      h[3] += mix64(ba ^ 0xd6e8feb86659fd93ull);
    }
    int64_t n0 = 0, e0 = 0, ng = N, eg = E;
    if (G > 0) {
      const int g = seg_hint = segment_of_hint(edge_off, G, e, seg_hint);
      n0 = node_off[g];
      e0 = edge_off[g];
      ng = node_off[g + 1] - n0;
      eg = edge_off[g + 1] - e0;
    }
    // every endpoint of a graph's entries lies in the graph's own node range: a list with an id outside it takes the
    // sorting build, which drops that entry (the sort-free placement k = e (+ s) would shift every later entry)
    if (s < n0 || s >= n0 + ng || d < n0 || d >= n0 + ng) {
      f[0] += 1u;
      f[1] += 1u;
    }
    const int64_t Ep = eg >= ng ? e0 + eg - ng : -1;   // end of the sorted prefix under the "+ loops" reading
    if (e + 1 < e0 + eg) {
      const int64_t s1 = (int64_t)ei[e + 1], d1 = (int64_t)ei[E + e + 1];
      const bool gt = s > s1 || (s == s1 && d > d1);
      f[0] += gt ? 1u : 0u;
      if (Ep >= 0 && e + 1 < Ep) f[1] += gt ? 1u : 0u;
      f[3] += (s == s1 && d == d1) ? 1u : 0u;
    }
    if (Ep < 0) f[2] += 1u;
    else if (e >= Ep) f[2] += (s == n0 + e - Ep && d == n0 + e - Ep) ? 0u : 1u;
  }
  __shared__ unsigned long long red[8][8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    unsigned long long v = q < 4 ? h[q] : f[q - 4];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    unsigned long long v = 0ull;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
    if (v) atomicAdd(out + threadIdx.x, v);   // integer sums: exact in any order
  }
}

template <typename IndexT>
static int csr_build_any(const IndexT* edge_index, int64_t E, int64_t N, int by,
                         int loop_mode, const mgcn_csr_t* out, int32_t* bad_index,
                         void* workspace, size_t* workspace_bytes, void* stream, int presorted = 0, int64_t G = 0,
                         const int32_t* node_off = nullptr, const int32_t* edge_off = nullptr) {
  MGCN_REQUIRE(G >= 0 && G < (1 << 24) && (G == 0 || (node_off && edge_off && presorted && by == 0)), MGCN_ERR_SHAPE);
  MGCN_REQUIRE(presorted >= 0 && presorted <= 6, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(presorted == 0 || loop_mode == 0, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(!((presorted & 3) == 2) || E >= N, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(G == 0 || (presorted & 3) == 2, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(by == 0 || by == 1, MGCN_ERR_SHAPE);
  MGCN_REQUIRE(loop_mode >= 0 && loop_mode <= 2, MGCN_ERR_SHAPE);
  const int64_t kMax = (int64_t(1) << 31) - (int64_t(1) << 20);
  MGCN_REQUIRE(E >= 0 && N >= 0 && E < kMax && N < kMax, MGCN_ERR_RANGE);
  const int64_t total = E + (loop_mode == 2 ? N : 0);
  MGCN_REQUIRE(total < kMax, MGCN_ERR_RANGE);

  // the query sizes for the caller's seg_cap when the structure is passed, else for the worst case
  const int64_t n_tasks_cap = N + (out ? out->seg_cap : 2 * total + 2) + 1;
  int64_t items = total > N ? total : N;  // the sort buffers also serve the row- and task-order sorts
  if (n_tasks_cap > items) items = n_tasks_cap;
  const int num_blocks = (int)ceil_div(items > 0 ? items : 1, kRsTile);
  const int64_t hist_len = (int64_t)256 * num_blocks;
  WorkspaceCarver ws(workspace);
  uint32_t* keys_a = ws.take<uint32_t>(items);
  uint32_t* keys_b = ws.take<uint32_t>(items);
  int32_t* vals_a = ws.take<int32_t>(items);
  int32_t* vals_b = ws.take<int32_t>(items);
  int32_t* block_hist = ws.take<int32_t>(hist_len);
  int64_t scan_len = hist_len > N + 1 ? hist_len : N + 1;
  if (n_tasks_cap > scan_len) scan_len = n_tasks_cap;
  int32_t* tile_sums = ws.take<int32_t>(scan_tiles(scan_len));
  int32_t* len_w = ws.take<int32_t>(n_tasks_cap);
  int32_t* wpos = ws.take<int32_t>(n_tasks_cap);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(out != nullptr && bad_index != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(out->n_rows == N && out->nnz_cap >= total && out->hub_threshold >= 1, MGCN_ERR_SHAPE);
  int32_t* rowptr = const_cast<int32_t*>(out->rowptr);
  int32_t* nbr = const_cast<int32_t*>(out->nbr);
  int32_t* perm = const_cast<int32_t*>(out->perm);
  int32_t* order = const_cast<int32_t*>(out->order);
  int32_t* hub_rows = const_cast<int32_t*>(out->hub_rows);
  int32_t* hub_seg0 = const_cast<int32_t*>(out->hub_seg0);
  int32_t* hub_count = const_cast<int32_t*>(out->hub_count);
  int32_t* seg_row = const_cast<int32_t*>(out->seg_row);
  int32_t* seg_beg = const_cast<int32_t*>(out->seg_beg);
  int32_t* seg_count = const_cast<int32_t*>(out->seg_count);
  int4* tasks = reinterpret_cast<int4*>(const_cast<int32_t*>(out->tasks));
  MGCN_REQUIRE(rowptr && hub_count && seg_count, MGCN_ERR_NULL);
  MGCN_REQUIRE(tasks == nullptr || N == 0 || (aligned16(tasks) && order != nullptr), MGCN_ERR_ALIGN);
  MGCN_REQUIRE(total == 0 || (nbr && perm), MGCN_ERR_NULL);
  MGCN_REQUIRE(E == 0 || edge_index != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(out->hub_cap == 0 || (hub_rows && hub_seg0), MGCN_ERR_NULL);
  MGCN_REQUIRE(out->seg_cap == 0 || (seg_row && seg_beg), MGCN_ERR_NULL);
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  MGCN_CHECK_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(int32_t) * (N + 1), st));
  MGCN_CHECK_CUDA(cudaMemsetAsync(hub_count, 0, sizeof(int32_t), st));
  MGCN_CHECK_CUDA(cudaMemsetAsync(seg_count, 0, sizeof(int32_t), st));
  MGCN_CHECK_CUDA(cudaMemsetAsync(bad_index, 0, sizeof(int32_t), st));
  if (total > 0) {
    // (a presorted list is counted by source: its prefix is indexed through these row starts; a symmetric list has
    // the same counts by target)
    MGCN_LAUNCH(k_make_keys<IndexT>, grid_for(total, 256), 256, 0, stream, edge_index, E, N, presorted ? 0 : by,
                loop_mode, total, presorted ? nullptr : keys_a, rowptr, bad_index);   // a sort-free build needs no keys
  }
  int rc = exclusive_scan_i32(rowptr, rowptr, N + 1, tile_sums, stream);
  if (rc != MGCN_OK) return rc;

  if (total > 0 && presorted) {
    // layout bits: 1 = sorted, 2 = sorted prefix + N trailing loops, +4 = repeated entries possible
    MGCN_LAUNCH(k_fill_presorted<IndexT>, grid_for(total, 256), 256, 0, stream, edge_index, E, N, by,
                (presorted & 3) == 2 ? 1 : 0, (presorted & 4) ? 1 : 0, (int)G, node_off, edge_off, rowptr, nbr, perm);
  } else if (total > 0) {
    const int32_t* sorted_pos = nullptr;
    rc = radix_sort_positions(keys_a, keys_b, vals_a, vals_b, total, (uint64_t)N, block_hist,
                              tile_sums, &sorted_pos, stream);
    if (rc != MGCN_OK) return rc;
    MGCN_LAUNCH(k_finalize<IndexT>, grid_for(total, 256), 256, 0, stream, edge_index, E, by, total,
                sorted_pos, rowptr, N, nbr, perm);
  }
  if (N > 0 && out->hub_cap > 0 && out->seg_cap > 0) {
    MGCN_LAUNCH(k_find_hubs, (int)ceil_div(N, 256), 256, 0, stream, rowptr, N, out->hub_threshold,
                hub_rows, hub_seg0, out->hub_cap, hub_count, seg_row, seg_beg, out->seg_cap,
                seg_count);
  }
  if (N > 0 && order != nullptr) {
    MGCN_LAUNCH(k_order_keys, (int)ceil_div(N, 256), 256, 0, stream, rowptr, N, keys_a);
    const uint64_t max_key =
        ((uint64_t)((N - 1) >> kOrderWindowShift) << kOrderLenBits) | ((1u << kOrderLenBits) - 1);
    const int32_t* sorted_rows = nullptr;
    rc = radix_sort_positions(keys_a, keys_b, vals_a, vals_b, N, max_key, block_hist, tile_sums,
                              &sorted_rows, stream);
    if (rc != MGCN_OK) return rc;
    MGCN_LAUNCH(k_copy_i32, (int)ceil_div(N, 256), 256, 0, stream, sorted_rows, N, order);
    if (tasks != nullptr) {
      int32_t* nbr_w = const_cast<int32_t*>(out->nbr_w);
      MGCN_REQUIRE(total == 0 || nbr_w != nullptr, MGCN_ERR_NULL);
      const bool hubs = out->hub_cap > 0 && out->seg_cap > 0;
      const int64_t seg_cap = hubs ? out->seg_cap : 0;
      const int32_t thr = hubs ? out->hub_threshold : 0x7fffffff;
      const int64_t n_tasks = N + seg_cap;
      MGCN_LAUNCH(k_task_keys, (int)ceil_div(n_tasks, 256), 256, 0, stream, rowptr, N, seg_row,
                  seg_count, seg_cap, keys_a);
      const uint64_t max_task_key =
          ((uint64_t)(((N - 1) >> kOrderWindowShift) + 1) << (kOrderLenBits + 1)) | (1u << kOrderLenBits);
      const int32_t* tid = nullptr;
      rc = radix_sort_positions(keys_a, keys_b, vals_a, vals_b, n_tasks, max_task_key, block_hist,
                                tile_sums, &tid, stream);
      if (rc != MGCN_OK) return rc;
      MGCN_LAUNCH(k_task_lengths, (int)ceil_div(n_tasks + 1, 256), 256, 0, stream, tid, rowptr, N,
                  seg_row, seg_beg, seg_count, seg_cap, thr, len_w);
      rc = exclusive_scan_i32(len_w, wpos, n_tasks + 1, tile_sums, stream);
      if (rc != MGCN_OK) return rc;
      MGCN_LAUNCH(k_make_tasks, (int)ceil_div(n_tasks * 8, 256), 256, 0, stream, tid, rowptr, N,
                  seg_row, seg_beg, seg_count, seg_cap, thr, wpos, nbr, tasks, nbr_w);
    }
  }
  return MGCN_OK;
}

extern "C" int mgcn_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int by,
                              int loop_mode, const mgcn_csr_t* out, int32_t* bad_index,
                              void* workspace, size_t* workspace_bytes, void* stream) {
  return csr_build_any<int64_t>(edge_index, E, N, by, loop_mode, out, bad_index, workspace, workspace_bytes, stream);
}

extern "C" int mgcn_csr_build_i32(const int32_t* edge_index, int64_t E, int64_t N, int by,
                                  int loop_mode, const mgcn_csr_t* out, int32_t* bad_index,
                                  void* workspace, size_t* workspace_bytes, void* stream) {
  return csr_build_any<int32_t>(edge_index, E, N, by, loop_mode, out, bad_index, workspace, workspace_bytes, stream);
}

extern "C" int mgcn_csr_build_presorted(const int64_t* edge_index, int64_t E, int64_t N, int by, int layout,
                                        int64_t G, const int32_t* node_off, const int32_t* edge_off,
                                        const mgcn_csr_t* out, int32_t* bad_index, void* workspace,
                                        size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(layout >= 1 && layout <= 6 && (layout & 3) != 0 && (layout & 3) != 3, MGCN_ERR_SHAPE);
  return csr_build_any<int64_t>(edge_index, E, N, by, 0, out, bad_index, workspace, workspace_bytes, stream, layout, G,
                                node_off, edge_off);
}

extern "C" int mgcn_csr_build_presorted_i32(const int32_t* edge_index, int64_t E, int64_t N, int by, int layout,
                                            int64_t G, const int32_t* node_off, const int32_t* edge_off,
                                            const mgcn_csr_t* out, int32_t* bad_index, void* workspace,
                                            size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(layout >= 1 && layout <= 6 && (layout & 3) != 0 && (layout & 3) != 3, MGCN_ERR_SHAPE);
  return csr_build_any<int32_t>(edge_index, E, N, by, 0, out, bad_index, workspace, workspace_bytes, stream, layout, G,
                                node_off, edge_off);
}

extern "C" int mgcn_degree_from_rowptr(const int32_t* rowptr, int64_t N, float* deg, void* stream) {
  MGCN_REQUIRE(N >= 0, MGCN_ERR_RANGE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(rowptr && deg, MGCN_ERR_NULL);
  MGCN_LAUNCH(k_degree, (int)ceil_div(N, 256), 256, 0, stream, rowptr, N, deg);
  return MGCN_OK;
}

extern "C" int mgcn_weighted_degree(const mgcn_csr_t* g, const float* edge_weight, int64_t E,
                                    float loop_weight, float* deg, void* stream) {
  MGCN_REQUIRE(g && deg, MGCN_ERR_NULL);
  if (g->n_rows == 0) return MGCN_OK;
  MGCN_REQUIRE(g->rowptr && g->perm, MGCN_ERR_NULL);
  MGCN_REQUIRE(E == 0 || edge_weight, MGCN_ERR_NULL);
  MGCN_LAUNCH(k_weighted_degree, (int)ceil_div(g->n_rows, 256), 256, 0, stream, g->rowptr, g->perm,
              edge_weight, E, loop_weight, g->n_rows, deg);
  return MGCN_OK;
}

namespace mgcn {
// Multiset fingerprint of the edge list and of its transpose: sums (mod 2^64) of two independent 64-bit mixes
// of (src, dst) resp. (dst, src).  Equal fingerprints <=> the directed edge multiset is symmetric (up to a
// 2^-128 collision chance), in which case the structure by source lists, row by row, the same neighbour
// multisets as the structure by target and need not be built.  Integer sums: independent of scheduling.
template <typename IndexT>
__global__ void __launch_bounds__(256) k_edge_fingerprint(const IndexT* __restrict__ ei, int64_t E,
                                                          unsigned long long* __restrict__ out) {
  unsigned long long f[4] = {0ull, 0ull, 0ull, 0ull};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    const uint64_t a = (uint64_t)(int64_t)ei[e], b = (uint64_t)(int64_t)ei[E + e];
    const uint64_t ab = a * 0x9e3779b97f4a7c15ull + b, ba = b * 0x9e3779b97f4a7c15ull + a;
    f[0] += mix64(ab);
    f[1] += mix64(ba);
    f[2] += mix64(ab ^ 0xd6e8feb86659fd93ull);
    f[3] += mix64(ba ^ 0xd6e8feb86659fd93ull);
  }
  __shared__ unsigned long long red[8][4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    unsigned long long v = f[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    unsigned long long v = 0ull;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
    atomicAdd(out + threadIdx.x, v);
  }
}
}  // namespace mgcn

template <typename IndexT>
static int edge_fingerprint_any(const IndexT* edge_index, int64_t E, uint64_t* out4, void* stream) {
  MGCN_REQUIRE(out4 != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(E >= 0 && E < (int64_t(1) << 31), MGCN_ERR_RANGE);
  MGCN_CHECK_CUDA(cudaMemsetAsync(out4, 0, 4 * sizeof(uint64_t), static_cast<cudaStream_t>(stream)));
  if (E == 0) return MGCN_OK;
  MGCN_REQUIRE(edge_index != nullptr, MGCN_ERR_NULL);
  int64_t blocks = ceil_div(E, 256 * 8);
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  MGCN_LAUNCH(k_edge_fingerprint<IndexT>, (unsigned)blocks, 256, 0, stream, edge_index, E,
              reinterpret_cast<unsigned long long*>(out4));
  return MGCN_OK;
}

extern "C" int mgcn_edge_fingerprint(const int64_t* edge_index, int64_t E, uint64_t* out4, void* stream) {
  return edge_fingerprint_any<int64_t>(edge_index, E, out4, stream);
}

extern "C" int mgcn_edge_fingerprint_i32(const int32_t* edge_index, int64_t E, uint64_t* out4, void* stream) {
  return edge_fingerprint_any<int32_t>(edge_index, E, out4, stream);
}

template <typename IndexT>
static int edge_layout_any(const IndexT* edge_index, int64_t E, int64_t N, int64_t G, const int32_t* node_off,
                           const int32_t* edge_off, uint64_t* out8, void* stream) {
  MGCN_REQUIRE(out8 != nullptr, MGCN_ERR_NULL);
  MGCN_REQUIRE(N >= 0 && G >= 0 && G < (1 << 24), MGCN_ERR_RANGE);
  MGCN_REQUIRE(G == 0 || (node_off && edge_off), MGCN_ERR_NULL);
  MGCN_REQUIRE(E >= 0 && E < (int64_t(1) << 31), MGCN_ERR_RANGE);
  MGCN_CHECK_CUDA(cudaMemsetAsync(out8, 0, 8 * sizeof(uint64_t), static_cast<cudaStream_t>(stream)));
  if (E == 0) return MGCN_OK;
  MGCN_REQUIRE(edge_index != nullptr, MGCN_ERR_NULL);
  int64_t blocks = ceil_div(E, 256 * 8);
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  MGCN_LAUNCH(k_edge_order_check<IndexT>, (unsigned)blocks, 256, 0, stream, edge_index, E, N, (int)G, node_off,
              edge_off, reinterpret_cast<unsigned long long*>(out8));
  return MGCN_OK;
}

extern "C" int mgcn_edge_layout(const int64_t* edge_index, int64_t E, int64_t N, int64_t G, const int32_t* node_off,
                                const int32_t* edge_off, uint64_t* out8, void* stream) {
  return edge_layout_any<int64_t>(edge_index, E, N, G, node_off, edge_off, out8, stream);
}

extern "C" int mgcn_edge_layout_i32(const int32_t* edge_index, int64_t E, int64_t N, int64_t G,
                                    const int32_t* node_off, const int32_t* edge_off, uint64_t* out8, void* stream) {
  return edge_layout_any<int32_t>(edge_index, E, N, G, node_off, edge_off, out8, stream);
}

extern "C" int mgcn_gcn_norm(const float* deg, int64_t N, int mode, float* dis, void* stream) {
  MGCN_REQUIRE(N >= 0, MGCN_ERR_RANGE);
  MGCN_REQUIRE(mode == 0 || mode == 1, MGCN_ERR_SHAPE);
  if (N == 0) return MGCN_OK;
  MGCN_REQUIRE(deg && dis, MGCN_ERR_NULL);
  MGCN_LAUNCH(k_gcn_norm, (int)ceil_div(N, 256), 256, 0, stream, deg, N, mode, dis);
  return MGCN_OK;
}

extern "C" int mgcn_permute_edge_values(const mgcn_csr_t* g, const float* vals_in, int64_t E,
                                        float loop_value, float* vals_out, void* stream) {
  MGCN_REQUIRE(g && vals_out, MGCN_ERR_NULL);
  if (g->nnz_cap == 0) return MGCN_OK;
  MGCN_REQUIRE(g->rowptr && g->perm, MGCN_ERR_NULL);
  MGCN_REQUIRE(E == 0 || vals_in, MGCN_ERR_NULL);
  MGCN_LAUNCH(k_permute_vals, grid_for(g->nnz_cap, 256), 256, 0, stream, g->perm, g->rowptr,
              g->n_rows, g->nnz_cap, vals_in, E, loop_value, vals_out);
  return MGCN_OK;
}

extern "C" int mgcn_preprocess_edges(const int64_t* edge_index, int64_t E, int64_t N, int undirected,
                                     int add_loops, int64_t cap, int64_t* out, int32_t* perm,
                                     float* deg, int64_t* count, int32_t* bad_index, void* workspace,
                                     size_t* workspace_bytes, void* stream) {
  MGCN_REQUIRE(workspace_bytes != nullptr, MGCN_ERR_NULL);
  const int64_t kMax = (int64_t(1) << 31) - (int64_t(1) << 20);
  MGCN_REQUIRE(E >= 0 && N >= 0 && N < kMax, MGCN_ERR_RANGE);
  const int64_t M = undirected ? 2 * E : E;
  MGCN_REQUIRE(M + (add_loops ? N : 0) < kMax, MGCN_ERR_RANGE);
  const int64_t items = M > 0 ? M : 1;
  const int num_blocks = (int)ceil_div(items, kRsTile);
  const int64_t hist_len = (int64_t)256 * num_blocks;
  WorkspaceCarver ws(workspace);
  uint32_t* keys_a = ws.take<uint32_t>(items);
  uint32_t* keys_b = ws.take<uint32_t>(items);
  int32_t* vals_a = ws.take<int32_t>(items);
  int32_t* vals_b = ws.take<int32_t>(items);
  int32_t* vals_c = ws.take<int32_t>(items);
  int32_t* block_hist = ws.take<int32_t>(hist_len);
  const int64_t scan_len = hist_len > M + 1 ? hist_len : M + 1;
  int32_t* tile_sums = ws.take<int32_t>(scan_tiles(scan_len));
  int32_t* flags = ws.take<int32_t>(M + 1);
  int32_t* idx = ws.take<int32_t>(M + 1);
  int32_t* degi = ws.take<int32_t>(N > 0 ? N : 1);
  if (workspace == nullptr) {
    *workspace_bytes = ws.bytes();
    return MGCN_OK;
  }
  MGCN_REQUIRE(*workspace_bytes >= ws.bytes(), MGCN_ERR_WORKSPACE);
  MGCN_REQUIRE(out && perm && deg && count && bad_index, MGCN_ERR_NULL);
  MGCN_REQUIRE(cap >= M + (add_loops ? N : 0), MGCN_ERR_SHAPE);
  MGCN_REQUIRE(E == 0 || edge_index != nullptr, MGCN_ERR_NULL);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MGCN_CHECK_CUDA(cudaMemsetAsync(bad_index, 0, sizeof(int32_t), st));
  MGCN_CHECK_CUDA(cudaMemsetAsync(degi, 0, sizeof(int32_t) * (N > 0 ? N : 1), st));
  const int32_t* pos = nullptr;
  if (M > 0) {
    // stable by col, then stable by row  =>  lexicographic (row, col), first occurrence first
    MGCN_LAUNCH(k_pre_keys, grid_for(M, 256), 256, 0, stream, edge_index, E, M, N, 1, nullptr, keys_a, bad_index);
    int rc = radix_sort_positions(keys_a, keys_b, vals_a, vals_b, M, (uint64_t)(N > 0 ? N - 1 : 0), block_hist,
                                  tile_sums, &pos, stream);
    if (rc != MGCN_OK) return rc;
    MGCN_CHECK_CUDA(cudaMemcpyAsync(vals_c, pos, sizeof(int32_t) * M, cudaMemcpyDeviceToDevice, st));
    MGCN_LAUNCH(k_pre_keys, grid_for(M, 256), 256, 0, stream, edge_index, E, M, N, 0, vals_c, keys_a, bad_index);
    rc = radix_sort_positions(keys_a, keys_b, vals_a, vals_b, M, (uint64_t)(N > 0 ? N - 1 : 0), block_hist,
                              tile_sums, &pos, stream, vals_c);
    if (rc != MGCN_OK) return rc;
  }
  MGCN_LAUNCH(k_pre_flags, grid_for(M + 1, 256), 256, 0, stream, edge_index, E, M, pos, flags);
  int rc = exclusive_scan_i32(flags, idx, M + 1, tile_sums, stream);
  if (rc != MGCN_OK) return rc;
  if (M > 0) {
    MGCN_LAUNCH(k_pre_compact, grid_for(M, 256), 256, 0, stream, edge_index, E, M, pos, flags, idx, cap, N, out, perm,
                degi);
  }
  MGCN_LAUNCH(k_pre_finish, grid_for(N > 0 ? N : 1, 256), 256, 0, stream, idx, M, N, add_loops, cap, out, perm, degi,
              deg, count);
  return MGCN_OK;
}
