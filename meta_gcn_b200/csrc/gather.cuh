// Row gather shared by the aggregation kernels (gcn_layer.cu, gcn_fwd_tc.cu, gate.cu).
#pragma once
#include "common.cuh"

namespace mgcn {

constexpr int kGH = 32;   // row width of the flat gather

// ---- row gather: 4 lanes x 256 bits per row ------------------------------------------------------
// A lane group of 4 lanes owns a row, each lane 8 of the 32 columns (one sm_100 LDG.256 per gathered
// row and lane), so a warp instruction fetches 8 rows.  Measured (scripts/ubench.cu, one-graph window,
// 4 CTAs/SM): 16.8 TB/s against 11.4 TB/s for 8 lanes x LDG.128 — half the load / shuffle / address
// instructions per gathered byte and twice the bytes in flight per warp.
// The entries of a row are summed in row order (= edge_index order), one rounded add per entry, 4
// gathers in flight per group; the index batch after next is fetched before the gathers are issued
// (the index stream nbr_w is sequential in work order).
#ifndef MGCN_GATHER_U
#define MGCN_GATHER_U 4   // row gathers in flight per lane group
#endif

struct Row8 {
  float v[8];
};

__device__ __forceinline__ Row8 ld_row8(const float* p) {
  Row8 r;
  // gathered rows do not allocate in L1: its hit rate on them is 8 % (ncu), and skipping the allocation is worth
  // 1 - 2 % of the gather kernels (L1::evict_last was slower, plain allocation the previous default)
#ifdef MGCN_GATHER_L1ALLOC
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#else
  asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#endif
               : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]),
                 "=f"(r.v[6]), "=f"(r.v[7])
               : "l"(p));
  return r;
}

// Experiment switch (default off): L2 prefetch of a row that a later round will gather — the lane that holds the
// index of entry k asks for that row's line while the current round is in flight.  Measured at the botnet batch: no
// gain (k_agg_flat 0.482 -> 0.485 ms, k_gcn_fwd_tc 0.677 -> 0.681 ms): the gather is not waiting on HBM misses, it runs
// at the rate the L2 slices deliver sectors (~11 TB/s here against a ~12.4 TB/s full-chip cap).
#ifndef MGCN_GATHER_PREFETCH
#define MGCN_GATHER_PREFETCH 0
#endif
__device__ __forceinline__ void prefetch_row_l2(const float* p) {
#if MGCN_GATHER_PREFETCH
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#endif
}

__device__ __forceinline__ void row8_add(Row8& acc, const Row8& b) {
  // four packed f32x2 adds (sm_100 FADD2): same IEEE result per element as eight scalar adds
#pragma unroll
  for (int q = 0; q < 8; q += 2) {
    asm("{\n .reg .b64 a0, b0;\n mov.b64 a0, {%0, %1};\n mov.b64 b0, {%2, %3};\n"
        " add.rn.f32x2 a0, a0, b0;\n mov.b64 {%0, %1}, a0;\n}\n"
        : "+f"(acc.v[q]), "+f"(acc.v[q + 1])
        : "f"(b.v[q]), "f"(b.v[q + 1]));
  }
}

// Sum rows m[nbr_w[k]] for k in [beg, end), in order, for the 8 columns of this lane.  The 4 lanes of
// a group call this together; gi holds nbr_w[beg + sub] and gi_n holds nbr_w[beg + 4 + sub].
// gathered row through L1 (allocating): for kernels that leave the L1 most of the SM's 228 KB (no operand stages in
// shared memory), where the ~840 hub source rows of a botnet graph (12.7 % of all gathered entries) can stay resident
__device__ __forceinline__ Row8 ld_row8_l1(const float* p) {
  Row8 r;
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]),
                 "=f"(r.v[6]), "=f"(r.v[7])
               : "l"(p));
  return r;
}

// Gate of an edge j -> i from two per-node scores (EdgeGateProj, gcn_base_models.py:322-369):
// sigmoid(a_j + t_i) with t_i = b_i + c formed once per row.  Every kernel that needs a gate forms it with this one
// function from the same two operands, so the gates of the forward and of both backward passes are the same bits.
// ex2.approx and one rounded reciprocal (a few ulp of fp32, relative): an IEEE exp / divide costs the gated forward
// layer kernel spills at its 80-register cap.
__device__ __forceinline__ float edge_gate(float a_j, float t_i) {
  return __frcp_rn(__fadd_rn(1.f, __expf(-__fadd_rn(a_j, t_i))));
}

// kGate: every gathered row is weighted by edge_gate(ab[j].x, gate_t) before it is added (one rounded multiply)
template <bool kL1 = false, bool kGate = false>
__device__ __forceinline__ Row8 gather_sum(const float* __restrict__ m, const int32_t* __restrict__ nbr_w,
                                           int beg, int end, int gi, int gi_n, int sub, int grp_lane0,
                                           unsigned gmask, int col, uint64_t pol,
                                           const float2* __restrict__ ab = nullptr, float gate_t = 0.f) {
  Row8 acc;
#pragma unroll
  for (int q = 0; q < 8; ++q) acc.v[q] = 0.f;
  // gated: two rows in flight instead of four (with four, the gated forward layer kernel spills at its 80 registers)
  constexpr int U = kGate ? 2 : MGCN_GATHER_U;
  int e = beg;
  while (e < end) {
    const int cnt = min(4, end - e);
    int gi_nn = 0;
    if (e + 8 + sub < end) gi_nn = ld_i32_hint(nbr_w + e + 8 + sub, pol);
    if (e + 4 + sub < end) prefetch_row_l2(m + (int64_t)gi_n * kGH);   // next round's row of this lane
#pragma unroll
    for (int t0 = 0; t0 < 4; t0 += U) {
      if (t0 < cnt) {
        int j[U];
#pragma unroll
        for (int u = 0; u < U; ++u) j[u] = __shfl_sync(gmask, gi, grp_lane0 + ((t0 + u) & 3));
        Row8 xv[U];
        float sa[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (t0 + u < cnt) xv[u] = kL1 ? ld_row8_l1(m + (int64_t)j[u] * kGH + col) : ld_row8(m + (int64_t)j[u] * kGH + col);
          if constexpr (kGate) {
            if (t0 + u < cnt) sa[u] = __ldg(&ab[j[u]].x);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (t0 + u < cnt) {
            if constexpr (kGate) {
              const float gt = edge_gate(sa[u], gate_t);
#pragma unroll
              for (int q = 0; q < 8; ++q) xv[u].v[q] = __fmul_rn(gt, xv[u].v[q]);
            }
            row8_add(acc, xv[u]);
          }
        }
      }
    }
    e += 4;
    gi = gi_n;
    gi_n = gi_nn;
  }
  return acc;
}

__device__ __forceinline__ void store_partial(float* __restrict__ partial, int slot, int col, const Row8& acc) {
  float* p = partial + (int64_t)(slot - 1) * kGH + col;
  *reinterpret_cast<float4*>(p) = make_float4(acc.v[0], acc.v[1], acc.v[2], acc.v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(acc.v[4], acc.v[5], acc.v[6], acc.v[7]);
}

// partial rows of a hub's segments, added left to right (after k_hub_reduce: one row)
__device__ __forceinline__ Row8 ld_partial(const float* p) {
  const float4 lo = *reinterpret_cast<const float4*>(p), hi = *reinterpret_cast<const float4*>(p + 4);
  Row8 r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}
__device__ __forceinline__ Row8 sum_partials(const float* __restrict__ partial, int s0, int ns, int col) {
  const float* p = partial + (int64_t)s0 * kGH + col;
  Row8 tot = ld_partial(p);
  for (int q = 1; q < ns; ++q) {
    const Row8 b = ld_partial(p + (int64_t)q * kGH);
    row8_add(tot, b);
  }
  return tot;
}

// acc += p[0 .. 4 rows) in row order, the four 256-bit loads issued before the first add.  One asm statement: the
// compiler otherwise sinks each load next to its add, and an in-order warp then waits a full latency per row.
__device__ __forceinline__ void row8_add4(Row8& acc, const float* p) {
  asm volatile(
      "{\n .reg .f32 a<8>, b<8>, c<8>, d<8>;\n .reg .b64 x0, x1, x2, x3, y0, y1, y2, y3;\n"
      " ld.global.nc.v8.f32 {a0,a1,a2,a3,a4,a5,a6,a7}, [%8];\n"
      " ld.global.nc.v8.f32 {b0,b1,b2,b3,b4,b5,b6,b7}, [%8+128];\n"
      " ld.global.nc.v8.f32 {c0,c1,c2,c3,c4,c5,c6,c7}, [%8+256];\n"
      " ld.global.nc.v8.f32 {d0,d1,d2,d3,d4,d5,d6,d7}, [%8+384];\n"
      " mov.b64 x0, {%0,%1}; mov.b64 x1, {%2,%3}; mov.b64 x2, {%4,%5}; mov.b64 x3, {%6,%7};\n"
      " mov.b64 y0, {a0,a1}; mov.b64 y1, {a2,a3}; mov.b64 y2, {a4,a5}; mov.b64 y3, {a6,a7};\n"
      " add.rn.f32x2 x0, x0, y0; add.rn.f32x2 x1, x1, y1; add.rn.f32x2 x2, x2, y2; add.rn.f32x2 x3, x3, y3;\n"
      " mov.b64 y0, {b0,b1}; mov.b64 y1, {b2,b3}; mov.b64 y2, {b4,b5}; mov.b64 y3, {b6,b7};\n"
      " add.rn.f32x2 x0, x0, y0; add.rn.f32x2 x1, x1, y1; add.rn.f32x2 x2, x2, y2; add.rn.f32x2 x3, x3, y3;\n"
      " mov.b64 y0, {c0,c1}; mov.b64 y1, {c2,c3}; mov.b64 y2, {c4,c5}; mov.b64 y3, {c6,c7};\n"
      " add.rn.f32x2 x0, x0, y0; add.rn.f32x2 x1, x1, y1; add.rn.f32x2 x2, x2, y2; add.rn.f32x2 x3, x3, y3;\n"
      " mov.b64 y0, {d0,d1}; mov.b64 y1, {d2,d3}; mov.b64 y2, {d4,d5}; mov.b64 y3, {d6,d7};\n"
      " add.rn.f32x2 x0, x0, y0; add.rn.f32x2 x1, x1, y1; add.rn.f32x2 x2, x2, y2; add.rn.f32x2 x3, x3, y3;\n"
      " mov.b64 {%0,%1}, x0; mov.b64 {%2,%3}, x1; mov.b64 {%4,%5}, x2; mov.b64 {%6,%7}, x3;\n}\n"
      : "+f"(acc.v[0]), "+f"(acc.v[1]), "+f"(acc.v[2]), "+f"(acc.v[3]), "+f"(acc.v[4]), "+f"(acc.v[5]), "+f"(acc.v[6]),
        "+f"(acc.v[7])
      : "l"(p)
      : "memory");
}

// One warp per hub row: the row's segment partials -> one row, in place in the hub's first slot.  The biggest
// hub of a botnet graph has ~230 segments; summed by one lane group with dependent loads it alone took 60 us
// per aggregation.  Here the 8 lane groups sum 8 contiguous runs of segments concurrently and the 8 run sums
// are added left to right (a fixed order: deterministic).
__device__ __forceinline__ Row8 hub_run_sum(const float* __restrict__ partial, int s0, int q0, int q1, int col) {
  Row8 run;
#pragma unroll
  for (int q = 0; q < 8; ++q) run.v[q] = 0.f;
  if (q0 >= q1) return run;
  const float* pp = partial + (int64_t)(s0 + q0) * kGH + col;
  int q = q0;
  for (; q + 4 <= q1; q += 4, pp += 4 * kGH) row8_add4(run, pp);
  for (; q < q1; ++q, pp += kGH) {
    const Row8 b = ld_row8(pp);
    row8_add(run, b);
  }
  return run;
}

}  // namespace mgcn
