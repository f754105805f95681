/*
 * mgcn.h — C-ABI of libmgcn.so: the B200 (sm_100a) message-passing engine that sits behind
 * meta-gcn's Python model API.
 *
 * The reference (jzhou316/meta-gcn) is pure Python and has no FFI; its seams on this path are two
 * Python call shapes (SURVEY.md §8b):
 *   primitive seam  scatter_(name, src, index, dim_size)            src/gcn_meta/models/common.py:37-66
 *                   NodeModelBase.degnorm_const(...)                src/gcn_meta/models/gcn_base_models.py:65-146
 *   layer seam      NodeModelAdditive.forward(x, edge_index, ...)   src/gcn_meta/models/gcn_base_models.py:199-243
 *                   GCNConv / SAGEConv / GINConv / global_mean_pool kernel/gcn.py:26-29, gin.py:41-44,
 *                                                                   graph_sage.py:26-29 (PyG 1.3 semantics)
 * Every entry point below names the reference call it replaces. INTEGRATION.md shows the
 * ctypes / torch.library binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it says "host".
 *   - the library allocates nothing and never synchronises: the caller owns inputs, outputs and
 *     workspace, and all work is enqueued on `stream` (a cudaStream_t passed as void*).
 *   - workspace query: call with workspace == NULL, the required bytes are written to
 *     *workspace_bytes and MGCN_OK is returned without launching anything.
 *   - return value: 0 = OK, < 0 = argument error (MGCN_ERR_*), > 0 = cudaError_t of a launch.
 *   - indices are int64 at the boundary (the reference's edge_index dtype) and int32 inside.
 *   - features are fp32, row-major, leading dimension = row width.
 */
#ifndef MGCN_H_
#define MGCN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGCN_VERSION 100

#define MGCN_OK 0
#define MGCN_ERR_NULL (-1)      /* a required pointer is NULL                         */
#define MGCN_ERR_RANGE (-2)     /* N or E outside [0, 2^31 - 2^20)                     */
#define MGCN_ERR_SHAPE (-3)     /* unsupported width / stride / enum value            */
#define MGCN_ERR_ALIGN (-4)     /* pointer not aligned for 128-bit access             */
#define MGCN_ERR_WORKSPACE (-5) /* workspace smaller than the queried size            */

/* Rows longer than this are "hubs": they are cut into segments of this many entries, each summed by
 * one lane group like an ordinary row (from 0, in row order).  Rows at or below it are summed by one
 * lane group sequentially in edge_index order (bit-identical to the reference's CPU scatter_add).
 * The ns segment sums p_0 .. p_{ns-1} of a hub are combined in one of two fixed orders:
 *   left to right       ((p_0 + p_1) + p_2) + ...            mgcn_spmm; mgcn_aggregate_prescaled except below
 *   runs                R_g = sum of p_{g*per} .. p_{min(ns, g*per+per)-1}, each from 0, left to right;
 *                       then ((R_0 + R_1) + R_2) + ... over the non-empty runs, with
 *                       per = ceil(ns/8) (8 runs) if ns <= 32, per = ceil(ns/64) (64 runs) if ns > 32
 *                       — mgcn_aggregate_prescaled at H = 32 without mean / bias / residual on a 32-byte
 *                       aligned x, and mgcn_gcn_layer_fwd
 *   8 runs              the same with per = ceil(ns/8) for every ns — the tcgen05 hidden-32 layer kernels
 *                       (mgcn_gcn_layer_fwd_tc*)
 * Each is independent of the grid, the device and the order of the hub table, so results are identical
 * from run to run and across devices; they give different bits for hubs of more than 2 segments. */
#define MGCN_DEFAULT_HUB_THRESHOLD 64

/* A row-owned adjacency (CSR when built by source, CSC when built by target).  All pointer members
 * are DEVICE buffers owned by the caller; mgcn_csr_build fills them.  Capacities come from
 * mgcn_csr_capacities. */
typedef struct mgcn_csr {
  int64_t n_rows;           /* N                                                               */
  int64_t nnz_cap;          /* length of nbr/perm: E, or E+N when loops are appended           */
  int64_t hub_cap;          /* length of hub_rows/hub_seg0                                     */
  int64_t seg_cap;          /* length of seg_row/seg_beg                                       */
  int32_t hub_threshold;    /* hub limit = segment length                                      */
  int32_t reserved;
  const int32_t* rowptr;    /* [N+1]; rowptr[N] = number of kept edges                         */
  const int32_t* nbr;       /* [nnz_cap] other endpoint of each kept edge, row-grouped         */
  const int32_t* perm;      /* [nnz_cap] position in the input edge_index (E+i = loop of i)    */
  const int32_t* order;     /* [N] rows sorted by (row / 16384, length): the work order that
                               keeps the rows sharing a warp equally long; may be NULL         */
  const int32_t* hub_rows;  /* [hub_cap] rows longer than hub_threshold                        */
  const int32_t* hub_seg0;  /* [hub_cap] first segment of each hub row                         */
  const int32_t* hub_count; /* [1]                                                             */
  const int32_t* seg_row;   /* [seg_cap] row of each segment                                   */
  const int32_t* seg_beg;   /* [seg_cap] first entry of each segment                           */
  const int32_t* seg_count; /* [1]                                                             */
  const int32_t* tasks;     /* [(N + seg_cap) * 4] work descriptors {row, beg, end, partial_slot}:
                               entries [0,N) are the rows in `order` (row = -1 for a hub row, which
                               is covered by its segments), entries [N, N+seg_count) are the hub
                               segments (partial_slot = segment index + 1); beg/end index nbr_w;
                               16-byte aligned; may be NULL (then the task-driven kernels —
                               mgcn_aggregate_prescaled, mgcn_gcn_layer_fwd — are unavailable)  */
  const int32_t* nbr_w;     /* [nnz_cap] nbr in WORK order: the entries of task s are
                               nbr_w[tasks[s].beg .. tasks[s].end) in row order, and task s+1 starts
                               where task s ends, so a kernel walking the tasks reads the index
                               stream sequentially; NULL iff tasks is NULL                      */
} mgcn_csr_t;

int mgcn_version(void);
const char* mgcn_error_string(int code);
/* kernels launched by this library in this process since load / last reset (host counters) */
int64_t mgcn_launch_count(void);
void mgcn_reset_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * edge_index -> row-owned structure.  Replaces the sort-free COO bookkeeping the reference leaves
 * to torch_scatter (common.py:56-59) and PyG's add_remaining_self_loops / remove_self_loops
 * (inside GCNConv.norm, SAGEConv.forward, GINConv.forward; Appendix A of SURVEY.md).
 *
 * edge_index: int64 [2,E] row-major (row 0 = source, row 1 = target; gcn_base_models.py:28-41).
 * by        : 0 = group by source (edge_index[0]), 1 = group by target (edge_index[1]).
 * loop_mode : 0 keep edges as given; 1 drop self loops (remove_self_loops);
 *             2 drop self loops then append one loop per node at the END of the edge list
 *               (add_remaining_self_loops without weights) — nnz_cap must be E+N.
 * The order of edges inside a row is their order in edge_index (stable LSD radix sort), which is
 * the order the reference's CPU scatter_add sums them in.
 * out: every pointer member is a caller-allocated device buffer of the capacity given by
 *      mgcn_csr_capacities; n_rows / capacities / hub_threshold are filled in by the caller.
 * bad_index int32[1] is set to 1 if any endpoint is outside [0,N) (such edges are dropped).
 * perm entries past rowptr[N] are -1.
 */
int mgcn_csr_capacities(int64_t E, int64_t N, int loop_mode, int32_t hub_threshold,
                        int64_t* nnz_cap, int64_t* hub_cap, int64_t* seg_cap);
int mgcn_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int by, int loop_mode,
                   const mgcn_csr_t* out, int32_t* bad_index, void* workspace,
                   size_t* workspace_bytes, void* stream);
/* the same for an edge_index stored as int32 [2,E] (converted once when the dataset is loaded): the botnet batch
 * ships 600 MB of int64 indices per step over PCIe (batch.to(device), train_botnet.py:282), 300 MB as int32 */
int mgcn_csr_build_i32(const int32_t* edge_index, int64_t E, int64_t N, int by, int loop_mode,
                       const mgcn_csr_t* out, int32_t* bad_index, void* workspace,
                       size_t* workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Edge preprocessing that defines the botnet edge order (SURVEY.md §8 f1): to_undirected_ey +
 * sort_unique_edges (data_procs/undirected.py:6-35: both directions, unique over row*N+col in lexicographic
 * (row, col) order, first occurrence kept), add_self_loops_ey (data_procs/loop.py:13-17: (i,i) for every
 * node appended at the END) and the out-degree feature (data_procs/data_add_degree.py:45-65, float32).
 * edge_index int64 [2,E]; out int64 [2,cap] (row 0 at out, row 1 at out+cap), cap >= (undirected ? 2E : E)
 * + (add_loops ? N : 0); count[0] = number of valid columns; perm[k] = index into the doubled edge list
 * (i < E: edge i, i >= E: edge i-E reversed) of the kept occurrence, -1 for appended loops; deg float[N].
 * Integer work: bit-exact and independent of scheduling. */
int mgcn_preprocess_edges(const int64_t* edge_index, int64_t E, int64_t N, int undirected, int add_loops,
                          int64_t cap, int64_t* out, int32_t* perm, float* deg, int64_t* count,
                          int32_t* bad_index, void* workspace, size_t* workspace_bytes, void* stream);

/* deg[i] = float(rowptr[i+1]-rowptr[i]): the unweighted scatter_add(ones, row) of
 * gcn_base_models.py:126 and data_procs/data_add_degree.py:60-63. */
int mgcn_degree_from_rowptr(const int32_t* rowptr, int64_t N, float* deg, void* stream);

/* Weighted degree: deg[i] = sum over the row's entries (in row order) of edge_weight[perm[k]]
 * (loop entries, perm >= E, contribute loop_weight).  gcn_base_models.py:126 with edge_weight. */
int mgcn_weighted_degree(const mgcn_csr_t* g, const float* edge_weight, int64_t E,
                         float loop_weight, float* deg, void* stream);

/* out4[0..3] = two independent 64-bit multiset fingerprints of the directed edge list, interleaved with the
 * same two of its transpose: out4[0] == out4[1] && out4[2] == out4[3] <=> every (u,v) occurs as often as (v,u).
 * The botnet data of the reference are symmetric by construction (data_procs/undirected.py:6-35); for such an
 * edge_index the structure by source (the transposed aggregation of the autograd, train_botnet.py:293) holds
 * the same neighbour multisets per row as the structure by target and is not built a second time. */
int mgcn_edge_fingerprint(const int64_t* edge_index, int64_t E, uint64_t* out4, void* stream);
int mgcn_edge_fingerprint_i32(const int32_t* edge_index, int64_t E, uint64_t* out4, void* stream);

/* Fingerprints plus the ORDER of the list, in one pass pair and one 64-byte result: out8[0..3] as mgcn_edge_fingerprint;
 * out8[4] = number of positions e with (src,dst)[e] > (src,dst)[e+1] over the whole list; out8[5] the same over the
 * first E-N entries; out8[6] = entries among the last N that are not the self loop (e-(E-N), e-(E-N)); out8[7] =
 * adjacent equal entries.  An entry with an endpoint outside [0, N) counts once in out8[4] and once in out8[5], so a
 * list holding one is never reported as ordered (mgcn_csr_build drops such an entry; the sort-free placement cannot).
 * If E < N, every entry counts in out8[6].  out8[4] == 0: the list is in (src,dst) order and its ids are in range;
 * out8[5] == 0 && out8[6] == 0: sorted prefix + the N loops appended at the end — the layout the reference's
 * preprocessing gives every botnet graph (data_procs/undirected.py:6-35: unique over row*N+col, sorted; loop.py:13-17:
 * loops at the END).
 * A BATCH of graphs (Batch.from_data_list, dataloader.py:11: the lists of G graphs one after the other, node ids
 * shifted) is described by node_off / edge_off int32 [G+1] (device; G = 0 and NULL: one graph): the order tests are
 * then made per graph (out8[4]: every graph's list sorted; out8[5], out8[6]: every graph = sorted prefix + its own
 * loops, counted over the graph's own E and N; no pair across a graph boundary is compared), and the range test is
 * against the graph's own node range. */
int mgcn_edge_layout(const int64_t* edge_index, int64_t E, int64_t N, int64_t G, const int32_t* node_off,
                     const int32_t* edge_off, uint64_t* out8, void* stream);
int mgcn_edge_layout_i32(const int32_t* edge_index, int64_t E, int64_t N, int64_t G, const int32_t* node_off,
                         const int32_t* edge_off, uint64_t* out8, void* stream);

/* mgcn_csr_build (loop_mode 0) for a list whose order the caller has established with mgcn_edge_layout — no sort:
 * layout 1 = sorted by (src,dst); 2 = sorted prefix + N trailing loops; + 4 if entries may repeat (out8[7] != 0).
 * by = 0 (source): any such list.  by = 1 (target): the list must also be symmetric (fingerprints equal); each
 * entry's place is then that of its mirror edge, found by a binary search in the mirror's row (one graph only).
 * G / node_off / edge_off as in mgcn_edge_layout (batches: by = 0, layout 2 or 6).  A batch whose graphs are each in
 * layout 1 (or 5) with in-range ids is in that layout as ONE list too — node ids ascend from graph to graph — and is
 * passed as one list (G = 0).  Same outputs, bit for bit, as
 * mgcn_csr_build; the botnet batch (37.5 M entries): 1.3 ms by source against 3.5 ms with the three radix passes. */
int mgcn_csr_build_presorted(const int64_t* edge_index, int64_t E, int64_t N, int by, int layout, int64_t G,
                             const int32_t* node_off, const int32_t* edge_off, const mgcn_csr_t* out,
                             int32_t* bad_index, void* workspace, size_t* workspace_bytes, void* stream);
int mgcn_csr_build_presorted_i32(const int32_t* edge_index, int64_t E, int64_t N, int by, int layout, int64_t G,
                                 const int32_t* node_off, const int32_t* edge_off, const mgcn_csr_t* out,
                                 int32_t* bad_index, void* workspace, size_t* workspace_bytes, void* stream);

/* dis = deg^-1/2 (mode 0, 'sm') or deg^-1 (mode 1, 'rw') with inf -> 0:
 * gcn_base_models.py:128-135.  Computed as correctly rounded 1/sqrt(d) resp. 1/d. */
int mgcn_gcn_norm(const float* deg, int64_t N, int mode, float* dis, void* stream);

/* vals_out[k] = perm[k] < E ? vals_in[perm[k]] : loop_value  — edge weights into row order. */
int mgcn_permute_edge_values(const mgcn_csr_t* g, const float* vals_in, int64_t E,
                             float loop_value, float* vals_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Row-owned aggregation (the hot kernel).  Replaces index_select -> mul -> scatter_add of
 * gcn_base_models.py:223-237 / MessagePassing.propagate, and its autograd (index_add_/gather)
 * when called with the structure built by the other endpoint.
 *
 *   w_k   = nbr_scale[nbr[k]] * edge_val[k] * row_scale[i]     (absent factors skipped; each product
 *                                                              rounded to fp32, left to right — the
 *                                                              order of gcn_base_models.py:138-139)
 *   acc_i = sum_k  x[nbr[k], :] * w_k                           (k in row order, mul and add rounded
 *                                                              separately: no FMA contraction)
 *   acc_i = acc_i / max(len_i, 1)                               if reduce == 1 (scatter_mean)
 *   out_i = act( acc_i + bias + residual_i )                    act: 0 none, 1 relu
 * x: [n_in, H], out/residual: [g->n_rows, H]; edge_val is in ROW order (see
 * mgcn_permute_edge_values).  If gather_perm != 0 the gathered row is x[perm[k]] instead of
 * x[nbr[k]] (scatter_add of per-edge messages src[E,H]: common.py:56-59).
 */
int mgcn_spmm(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, int gather_perm,
              const float* edge_val, const float* nbr_scale, const float* row_scale, int reduce,
              const float* bias, const float* residual, int act, float* out, void* workspace,
              size_t* workspace_bytes, void* stream);

/* The same aggregation for inputs that already carry the per-source factor (x~ = nbr_scale * x,
 * written by the producing transform): no per-edge weight at all,
 *   out_i = act( post_scale[i] * sum_k x~[nbr[k], :] (/ len_i) + bias + residual_i ),
 * rows visited in g->order.  Same summation order as mgcn_spmm inside rows and hub segments; differs from it in
 * where the factors are rounded (x*(d_i d_j) vs (x d_j) summed, then * d_i) and, at H = 32 without reduce / bias /
 * residual on a 32-byte aligned x, in the combine order of hub segments ("runs", see MGCN_DEFAULT_HUB_THRESHOLD).
 * Epilogue order: * post_scale, / max(len_i, 1), + bias, + residual, act.  H must be 16, 32, 64 or 128; x, out,
 * bias and residual 16-byte aligned (else MGCN_ERR_ALIGN). */
int mgcn_aggregate_prescaled(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H,
                             const float* post_scale, int reduce, const float* bias,
                             const float* residual, int act, float* out, void* workspace,
                             size_t* workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dense transform on the FMA pipes (narrow widths) — torch.matmul(x, weight_node)
 * (gcn_base_models.py:201) and nn.Linear (gcn_model.py:64,73,96).
 *   y[n,c] = act( sum_k x[n,k] * W(k,c) + bias[c] + add[n,c] ),  W(k,c) = w[k*w_sk + c*w_sc]
 * so weight_node [Hi,Ho] uses (w_sk,w_sc)=(Ho,1) and nn.Linear.weight [Ho,Hi] uses (1,Hi);
 * the input-gradient dX = dY * W^T is the same call with the strides swapped.
 */
int mgcn_linear(const float* x, int64_t N, int64_t Hi, const float* w, int64_t w_sk, int64_t w_sc,
                int64_t Ho, const float* bias, const float* add, int act, float* y, void* stream);

/* mgcn_linear with two fused extras used by the whole-model path:
 *   xmask [N,Hi] (may be NULL): the operand is x * (xmask > 0)  — relu backward folded into the load
 *   row_scale [N] (may be NULL): y[n,:] = row_scale[n] * act(...) — messages leave pre-scaled by
 *   the per-source degree factor, so the aggregation needs no per-edge weight. */
int mgcn_linear_ex(const float* x, const float* xmask, int64_t N, int64_t Hi, const float* w,
                   int64_t w_sk, int64_t w_sc, int64_t Ho, const float* bias, const float* add,
                   int act, const float* row_scale, float* y, void* stream);

/* dW(k,c) = sum_n x[n,k] * g[n,c]  (written at dw[k*dw_sk + c*dw_sc]),  db[c] = sum_n g[n,c].
 * Two-stage fixed-order reduction: deterministic, no atomics.  db may be NULL. */
int mgcn_linear_wgrad(const float* x, int64_t N, int64_t Hi, const float* g, int64_t Ho, float* dw,
                      int64_t dw_sk, int64_t dw_sc, float* db, void* workspace,
                      size_t* workspace_bytes, void* stream);

/* The same transform for wide outputs on the 5th-generation tensor cores (tcgen05.mma, accumulators in
 * tensor memory): Ho in {64,128,192,256}, Hi % 4 == 0.  SAGEConv / GCNConv `matmul(x, weight) (+ bias)`
 * at hidden >= 64 (kernel/graph_sage.py:10,13; kernel/gcn.py:10,13; PyG 1.3 update()).  fp32 parity
 * through 3xTF32 with separately accumulated correction terms.  workspace holds the pre-split weight. */
int mgcn_linear_wide(const float* x, int64_t N, int64_t Hi, const float* w, int64_t w_sk, int64_t w_sc,
                     int64_t Ho, const float* bias, const float* add, int act, const float* row_scale,
                     float* y, void* workspace, size_t* workspace_bytes, void* stream);

/* mgcn_linear_wgrad with the gradient operand masked: g * (gmask > 0)  (gmask [N,Ho], may be NULL) */
int mgcn_linear_wgrad_ex(const float* x, int64_t N, int64_t Hi, const float* g, const float* gmask,
                         int64_t Ho, float* dw, int64_t dw_sk, int64_t dw_sc, float* db,
                         void* workspace, size_t* workspace_bytes, void* stream);

/* out[n,c] = row_scale[n] * g[n,c] * (m1[n,c] > 0) * (m2[n,c] > 0); masks and scale may be NULL.
 * H must be a multiple of 4.  (gradient entering the transposed aggregation: both ReLU masks of
 * a GCNModel layer and the per-node degree factor in one pass) */
int mgcn_masked_scale(const float* g, const float* m1, const float* m2, const float* row_scale,
                      int64_t N, int64_t H, float* out, void* stream);

/* g_in[n,c] = relu'(y[n,c]) * g[n,c]  (y = saved activation output; mask is y > 0). */
int mgcn_relu_backward(const float* g, const float* y, int64_t count, float* g_in, void* stream);

/* ---------------------------------------------------------------------------------------------
 * One residual GCN layer of the botnet model at hidden width 32 — GCNModel.forward's loop body
 * (gcn_model.py:89-106) around NodeModelAdditive.forward (gcn_base_models.py:199-243), and its
 * autograd (train_botnet.py:293), as fused launches.  m = pre * (x W_n) are the layer's messages,
 * already scaled by the per-source degree factor by whoever produced them (the previous layer's
 * launch, or mgcn_linear_ex for the first layer).
 *
 * forward:   h      = relu( post * sum_{e: col[e]=i} m[row[e]] + bias )     rows of g (built by target)
 *            y      = h + x res_w^T + res_b       (or h + resid when the residual term is precomputed:
 *                                                  first layer, input width != 32; exactly one of
 *                                                  x / resid is non-NULL)
 *            x_next = act_out ? relu(y) : y
 *            m_next = pre * (x_next w_next)       (w_next may be NULL: last layer)
 *            hmask[i] bit c = (h[i,c] > 0)
 * Sums run in edge_index order per row (hub rows: per segment, segments combined in runs — see
 * MGCN_DEFAULT_HUB_THRESHOLD); the dense
 * products run on the tensor pipe as 3xTF32 with separately accumulated correction terms.
 * Row-local mode, g == NULL: m[i] is the finished pre-activation of row i (n_in rows) — used for a first
 * layer of small input width, which is aggregated BEFORE its transform: (A_hat x) W instead of A_hat (x W).
 */
int mgcn_gcn_layer_fwd(const mgcn_csr_t* g, const float* m, int64_t n_in, const float* x,
                       const float* resid, const float* res_w, const float* res_b,
                       const float* w_next, const float* bias, const float* pre, const float* post,
                       int act_out, int64_t H, float* x_next, float* m_next, uint32_t* hmask,
                       void* workspace, size_t* workspace_bytes, void* stream);

/* First layer of the stack when its input is narrow (H_in <= 4; the botnet model feeds x = ones[N,1],
 * train_botnet.py:286): the layer is aggregated BEFORE its transform — s = sum_j pre_j x_j by mgcn_spmm on
 * [N,H_in] — and this launch forms, reading only s and x,
 *     h = relu(post * (s W_in)),  y = h + x R^T + r,  x' = act(y),  m' = pre * (x' W_next),  hmask = bits(h > 0)
 * i.e. NodeModelAdditive.forward (gcn_base_models.py:199-243) + the residual Linear / ReLU of gcn_model.py:96-105
 * for layer 0 without materialising x W_in or x R^T.  w_in [H_in][32] (in,out), res_w [32][H_in] (out,in). */
int mgcn_gcn_first_layer_fwd(const float* s, const float* x, int64_t N, int64_t Hin, const float* w_in,
                             const float* res_w, const float* res_b, const float* w_next, const float* pre,
                             const float* post, const float* out_scale, int act_out, int64_t H, float* x_next,
                             float* m_next, uint32_t* hmask, void* stream);
/* out_scale [N] (may be NULL; only with w_next == NULL): x_next rows leave multiplied by it — the input format of
 * mgcn_gcn_layer_fwd_tc below. */
/* The same with dropout on h (gcn_model.py:92, before the residual add): keep uint32 [N] = this layer's slice of
 * mgcn_dropout_keep_bits (one word per row, H = 32), keep_scale = 1 / (1 - p):
 *     h = bit c of keep[i] ? h * keep_scale : 0   (one rounded fp32 multiply);   hmask bit c = (h > 0) — kept and active
 * keep == NULL: exactly mgcn_gcn_first_layer_fwd.  keep needs w_next == NULL (the streaming pass); else MGCN_ERR_SHAPE. */
int mgcn_gcn_first_layer_fwd_ex(const float* s, const float* x, int64_t N, int64_t Hin, const float* w_in,
                                const float* res_w, const float* res_b, const float* w_next, const float* pre,
                                const float* post, const float* out_scale, const uint32_t* keep, float keep_scale,
                                int act_out, int64_t H, float* x_next, float* m_next, uint32_t* hmask, void* stream);
/* The same with the node-model bias (NodeModelAdditive's default bias=True; gcn_base_models.py:241), bias [32]:
 *     h = relu(post * (s W_in) + bias)   (one rounded fp32 add after the post multiply, then the ReLU, then dropout)
 * bias == NULL: exactly mgcn_gcn_first_layer_fwd_ex.  Both the streaming pass and the tile kernel take it. */
int mgcn_gcn_first_layer_fwd_bias(const float* s, const float* x, int64_t N, int64_t Hin, const float* w_in,
                                  const float* res_w, const float* res_b, const float* bias, const float* w_next,
                                  const float* pre, const float* post, const float* out_scale, const uint32_t* keep,
                                  float keep_scale, int act_out, int64_t H, float* x_next, float* m_next,
                                  uint32_t* hmask, void* stream);

/* One residual GCN layer forward at hidden 32, AGGREGATE-THEN-TRANSFORM, on tcgen05.mma / tensor memory
 * (csrc/gcn_fwd_tc.cu) — the default of the hidden-32 stack.  Same reference lines as mgcn_gcn_layer_fwd
 * (gcn_model.py:89-106, gcn_base_models.py:199-243), computed as (A_hat x) W instead of A_hat (x W):
 *     s_i    = post_i * sum_{e: col[e]=i} z[row[e]]          z = in_scale (.) x_n: the stored rows carry the
 *                                                            per-source degree factor, so no per-edge weight is read
 *     h_i    = relu(s_i w + bias);   hmask[i] bit c = (h[i,c] > 0)
 *     y_i    = h_i + (z_i res_w^T) / in_scale_i + res_b      (= h_i + x_i res_w^T + res_b)
 *     z_next = out_scale_i * (act_out ? relu(y_i) : y_i)
 * The layer reads one [N,32] array and writes one (no message array beside the activations).  in_scale / post /
 * out_scale are [N] or NULL (= 1); in_scale must be > 0 on every row (callers store sigma = pre where pre > 0, else 1:
 * a row with pre == 0 computed from the graph's own out-degree is never gathered).  w [32][32] (in,out), res_w [32][32]
 * (out,in).  Sums run in edge_index order per row; dense products are 3xTF32 with separately accumulated corrections. */
int mgcn_gcn_layer_fwd_tc(const mgcn_csr_t* g, const float* z, int64_t n_in, const float* w, const float* res_w,
                          const float* res_b, const float* bias, const float* in_scale, const float* post,
                          const float* out_scale, int act_out, int64_t H, float* z_next, uint32_t* hmask,
                          void* workspace, size_t* workspace_bytes, void* stream);
/* The same layer with dropout on h, applied in the epilogue (hub rows included): keep uint32 [N] = this layer's slice of
 * mgcn_dropout_keep_bits, keep_scale = 1 / (1 - p):
 *     h_i = bit c of keep[i] ? h_i * keep_scale : 0   (one rounded fp32 multiply, as torch's dropout);  hmask bit c = (h > 0)
 * so the mask word carries kept * relu'(h) and the backward entry points need no change: the caller multiplies the
 * `post` it passes to them by keep_scale.  keep == NULL: exactly mgcn_gcn_layer_fwd_tc. */
int mgcn_gcn_layer_fwd_tc_ex(const mgcn_csr_t* g, const float* z, int64_t n_in, const float* w, const float* res_w,
                             const float* res_b, const float* bias, const float* in_scale, const float* post,
                             const float* out_scale, const uint32_t* keep, float keep_scale, int act_out, int64_t H,
                             float* z_next, uint32_t* hmask, void* workspace, size_t* workspace_bytes, void* stream);
/* The same layer with an edge gate (EdgeGateProj, gcn_base_models.py:322-369) on every gathered row:
 *     s_i = post_i * sum_{e: col[e]=i} g_e z[row[e]],   g_e = sigmoid(a_j + (b_i + c))   (j = row[e])
 * gate_ab float2 [n_in] = per-node scores (a, b) from mgcn_gate_scores, gate_c [1] = the gate bias on the device (NULL =
 * 0).  A gate is formed from the two endpoints while the row is gathered: no [E] array, no edge ids; hub segments are
 * gated before their partials are stored.  Everything after the gather is the contract of mgcn_gcn_layer_fwd_tc_ex.
 * gate_ab == NULL: exactly mgcn_gcn_layer_fwd_tc_ex (gate_c unused).  No allocation, capture-safe. */
int mgcn_gcn_layer_fwd_tc_gate(const mgcn_csr_t* g, const float* z, int64_t n_in, const float* w, const float* res_w,
                               const float* res_b, const float* bias, const float* in_scale, const float* post,
                               const float* out_scale, const uint32_t* keep, float keep_scale, const float* gate_ab,
                               const float* gate_c, int act_out, int64_t H, float* z_next, uint32_t* hmask,
                               void* workspace, size_t* workspace_bytes, void* stream);

/* backward, row-local part of layer n (dxw = pre * A^T gs comes from mgcn_aggregate_prescaled on the
 * structure built by source):
 *   G = dxw w^T + gy res_w;  dw = x^T dxw;  d_res_w = gy^T x;  d_res_b = colsum(gy)
 *   gy_prev = G * (x > 0);   gs_prev = post * gy_prev * bits(hmask_prev)      (both NULL: not wanted)
 * Weight gradients are reduced in a fixed order (deterministic, no atomics).
 * Runs on tcgen05.mma / tensor memory.  Every operand is split once into tf32 hi/lo images in shared memory (K-major
 * images for the row-local products, SWIZZLE_128B_BASE32B images for the transposed ones); a persistent CTA per SM
 * runs producer / issuer / epilogue roles over two operand stages and two accumulator buffers (csrc/gcn_layer_tc.cu).
 * 0.58 ms per layer at the botnet batch (profiles/r1b_layer_summary.md).
 * x_scale [N] or NULL: the array passed as x holds x_scale (.) x (the stored format of mgcn_gcn_layer_fwd_tc); the
 * factor is divided out as the rows are loaded. */
int mgcn_gcn_layer_bwd_tc(const float* dxw, const float* gy, const float* x, const float* x_scale, const float* w,
                          const float* res_w, const uint32_t* hmask_prev, const float* post, int64_t N,
                          int64_t H, float* gy_prev, float* gs_prev, float* dw, float* d_res_w,
                          float* d_res_b, void* workspace, size_t* workspace_bytes, void* stream);
/* The same with the gradient of the node-model bias of the layer.  With gy = the gradient of the layer's output
 * before its activation (the gy above), hmask_cur = this layer's mask words (bit c = relu'(h) & kept) and
 * bias_scale = the dropout scale 1 / (1 - p) (1 without dropout):
 *     d_bias[c] = bias_scale * sum_i (bit c of hmask_cur[i]) * gy[i,c]
 * The per-target factor post does not enter it (d_bias is not a column sum of gs: post may be 0).  Computed after the
 * row-local launch by the pass of mgcn_mask_bits_colsum (two more launches, one more read of gy: summed inside the
 * row-local kernel it spills), in a fixed order, so it is identical from run to run; every other output is
 * bit-identical to mgcn_gcn_layer_bwd_tc.  d_bias == NULL: exactly mgcn_gcn_layer_bwd_tc (hmask_cur and bias_scale
 * unused); d_bias needs hmask_cur (else MGCN_ERR_NULL).  The workspace is larger with d_bias (query with the same
 * arguments). */
int mgcn_gcn_layer_bwd_tc_ex(const float* dxw, const float* gy, const float* x, const float* x_scale, const float* w,
                             const float* res_w, const uint32_t* hmask_prev, const uint32_t* hmask_cur,
                             const float* post, float bias_scale, int64_t N, int64_t H, float* gy_prev,
                             float* gs_prev, float* dw, float* d_res_w, float* d_res_b, float* d_bias,
                             void* workspace, size_t* workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Edge gates of the hidden-32 stack (csrc/gate.cu; EdgeGateProj, gcn_base_models.py:322-369, with in_edgedim None).
 * The gate of an edge j -> i depends on its endpoints only: g_ij = sigmoid(a_j + (b_i + c)) with per-node scores
 *     a_j = (x_j w) . u,   b_i = (x_i w) . v            (u = linsrc.weight[0], v = lintgt.weight[0], c = the gate bias)
 * Every entry point forms g from the same operands in the same order, so all of them see the same gate bits.
 * Sums run in edge_index order per row (hub rows: segment partials added in a fixed order): deterministic, no atomics.
 *
 * Scores: ab[i] = ((x_i . (w u)) / in_scale_i, (x_i . (w v)) / in_scale_i) as float2 [N] (w u formed per block in a fixed
 * order).  x [N,H] with H <= 32 (H = 32 for the stored z = in_scale (.) x of the stack, in_scale [N] or NULL = 1);
 * w [H][32] (in,out), u / v [32].  One launch, no workspace, capture-safe. */
int mgcn_gate_scores(const float* x, int64_t N, int64_t H, const float* in_scale, const float* w, const float* u,
                     const float* v, float* ab, void* stream);
/* Gated aggregation of a narrow input (H <= 4: the first layer, aggregated before its transform):
 *     out_i = sum_{e: col[e]=i} g_e x[row[e]]       over g's rowptr / nbr (row order = edge_index order)
 * ab / c as above (c NULL = 0).  One warp per row, lane-strided partial sums added in a fixed tree order.  One launch,
 * capture-safe. */
int mgcn_gate_spmm_narrow(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, const float* ab,
                          const float* c, float* out, void* stream);
/* Backward of the gate, by target (g = the structure of the forward, grouped by target).  gs [N,32] = the masked,
 * post-scaled gradient of the layer (mgcn_mask_bits_scale), m [N,32] = z w (= pre_j x_j w: the message before its gate):
 *     dt_ij = <gs_i, m_j> * g_ij (1 - g_ij)                     (the gradient at the sigmoid's input)
 *     db_i  = sum_{j: j->i} dt_ij                               -> db [N]
 * Workspace: one float per hub segment (query with workspace == NULL).  Two launches with hub rows, else one;
 * no allocation, capture-safe. */
int mgcn_gate_grad_by_target(const mgcn_csr_t* g, const float* gs, const float* m, const float* ab, const float* c,
                             float* db, void* workspace, size_t* workspace_bytes, void* stream);
/* Backward of the gated aggregation by source (gt = grouped by source; the forward's structure when it is symmetric).
 * With dt_ij computed exactly as in mgcn_gate_grad_by_target (the same bits) and db from it:
 *     da_j  = sum_{i: j->i} dt_ij
 *     dxw_j = pre_j * sum_{i: j->i} g_ij gs_i + da_j u + db_j v     (= dL / d(x_j w); pre NULL = 1)
 *     dsc_j = (da_j / sigma_j, db_j / sigma_j, db_j)                 (sigma NULL = 1) -> dsc [N,3]
 * so that [du | dv] = m^T dsc[:, 0:2] and dc = colsum(dsc[:, 2]) (one mgcn_linear_wgrad).  dxw enters
 * mgcn_gcn_layer_bwd_tc(_ex) as the transposed aggregation would.  Workspace: one [33] float row per hub segment.
 * Two launches with hub rows, else one; no allocation, capture-safe. */
int mgcn_gate_grad_by_source(const mgcn_csr_t* gt, const float* gs, const float* m, const float* ab, const float* c,
                             const float* db, const float* pre, const float* u, const float* v, const float* sigma,
                             float* dxw, float* dsc, void* workspace, size_t* workspace_bytes, void* stream);

/* gs[i,c] = post[i] * gy[i,c] * bit c of bits[i]   (H = 32; post may be NULL) */
int mgcn_mask_bits_scale(const float* gy, const uint32_t* bits, const float* post, int64_t N,
                         int64_t H, float* gs, void* stream);

/* d_bias[c] = scale * sum_i (bit c of bits[i]) * gy[i,c]   (H = 32): the node-model bias gradient of a layer without a
 * row-local backward launch (the narrow-input first layer), the formula of mgcn_gcn_layer_bwd_tc_ex.  Per-block partial
 * sums over a grid that depends on N only, then one block adds them in a fixed order: identical from run to run.
 * N == 0 writes zeros.  Two launches; workspace query as elsewhere (workspace == NULL). */
int mgcn_mask_bits_colsum(const float* gy, const uint32_t* bits, float scale, int64_t N, int64_t H, float* d_bias,
                          void* workspace, size_t* workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dropout keep masks of the residual stack — nn.Dropout(p) of gcn_model.py:92 on every layer's h, as bits.
 * keep uint32 [L][N][W] (W words per row, W >= ceil(H/32)); bit b of keep[l][n][w] = column 32w + b of row n in layer l
 * is kept.  A pure function of (seed, l, n, column), independent of the launch configuration:
 *   key      (k0, k1) = (low 32 bits, high 32 bits) of seed[0] (ONE int64 in device memory: drawn on the device, so a
 *            captured CUDA graph draws anew on every replay)
 *   calls    for j = 0..3:  (r0, r1, r2, r3) = Philox4x32-10(counter = (n, l, 4w + j, 0), key)
 *   draws    r_i & 0xffff is column 32w + 8j + 2i, r_i >> 16 is column 32w + 8j + 2i + 1
 *   rule     kept iff draw >= t, t = nearest integer to p * 65536 (ties to even)
 * The keep probability is 1 - t / 65536, within 2^-17 of 1 - p (exact for p = k / 65536, e.g. 0.5); 16-bit draws
 * give 4 Philox calls per 32-column word instead of 8.  p outside [0, 1] or t = 65536 (nothing kept): MGCN_ERR_SHAPE.
 * One launch for all L layers. */
int mgcn_dropout_keep_bits(const int64_t* seed, int64_t L, int64_t N, int64_t W, float p, uint32_t* keep,
                           void* stream);
/* h[n,c] = bit (c % 32) of keep[n*W + c/32] ? h[n,c] * scale : 0, in place (H % 4 == 0, W >= ceil(H/32)): dropout on the
 * saved h of the generic stack (widths 16..128); its ReLU mask is then h > 0. */
int mgcn_dropout_apply(float* h, const uint32_t* keep, int64_t N, int64_t H, int64_t W, float scale, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Segment reductions — global_mean_pool / global_add_pool (kernel/gcn.py:29, gin.py:44,
 * graph_sage.py:29) and GCNModel's pred_on='graph' mean (gcn_model.py:112-123).
 * offsets int32[G+1] delimit contiguous node ranges (batch vector sorted ascending).
 */
int mgcn_batch_to_offsets(const int64_t* batch, int64_t N, int64_t G, int32_t* offsets, void* stream);
/* out[g,:] = sum (mode 0) or mean with count clamped to >= 1 (mode 1) of x[offsets[g]:offsets[g+1],:].
 * N = offsets[G] (total rows, host value: decides how many CTAs share a long segment).  Segments of up to
 * 64 rows are summed in row order (the reference's scatter order); longer ones in fixed contiguous chunks. */
int mgcn_segment_reduce(const float* x, int64_t H, const int32_t* offsets, int64_t G, int64_t N, int mode,
                        float* out, void* workspace, size_t* workspace_bytes, void* stream);
/* dx[n,:] = gout[g(n),:] (mode 0) or gout[g(n),:] / max(len_g,1) (mode 1) */
int mgcn_segment_broadcast(const float* gout, int64_t H, const int32_t* offsets, int64_t G,
                           int64_t N, int mode, float* dx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * BatchNorm1d — the last stage of the GIN convolution's MLP (kernel/gin.py:10-16: Sequential(Linear, ReLU, Linear,
 * ReLU, BatchNorm1d(hidden)); torch defaults eps 1e-5, momentum 0.1, affine).  x, y, g, dx: [N,H] row-major.
 * training != 0: batch statistics (two passes: mean, then centred second moment), running_mean / running_var updated
 * in place (unbiased variance, as torch does; either may be NULL); training == 0: the running statistics are used.
 * mean [H] / rstd [H] are outputs of the forward and inputs of the backward.  gamma / beta may be NULL (no affine).
 * backward: dbeta = colsum(g), dgamma = colsum(g * xhat), dx = gamma rstd (g - dbeta/N - xhat dgamma/N) in training
 * mode, gamma rstd g in evaluation mode (dx may be NULL).  Fixed-order reductions: deterministic, no atomics. */
int mgcn_batchnorm_fwd(const float* x, int64_t N, int64_t H, const float* gamma, const float* beta, float eps,
                       float momentum, int training, float* running_mean, float* running_var, float* mean,
                       float* rstd, float* y, void* workspace, size_t* workspace_bytes, void* stream);
int mgcn_batchnorm_bwd(const float* x, const float* g, int64_t N, int64_t H, const float* gamma, const float* mean,
                       const float* rstd, int training, float* dx, float* dgamma, float* dbeta, void* workspace,
                       size_t* workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Node-level cross entropy — nn.CrossEntropyLoss()(x, batch.y.long()) (train_botnet.py:225,287).
 * loss[0] = sum_n ( logsumexp(logits[n,:]) - logits[n, target[n]] ) (* 1/N if mean), fixed-order
 * two-stage sum.  A row's NLL is log1p(t) - (z_y - m), m = max_c z_c, t = sum of exp(z_c - m) over the classes
 * other than the first maximal one, so a confidently classified row keeps its small loss.
 * bwd: dlogits = (softmax - onehot) * (1/N if mean) * upstream[0]   (upstream: device scalar or NULL); the label's
 * entry is computed as -(sum over c != y of exp(z_c - m)) / s, not p_y - 1.
 *
 * Labels (both cross-entropy contracts, this one and the fused head below): a label outside [0, C) — -100
 * included, which is not an "ignore" value here — makes loss[0] NaN in both reductions, makes that row's
 * gradient NaN (its dlogits row; in the fused head its dx row and so dw and db), and is skipped by the counters.
 * bad_target int32[1] is set when such a label occurs.  No host synchronisation is involved.
 * No rows (N = 0): the sum is 0, the mean NaN (as torch); gradients over no rows are 0.
 */
int mgcn_cross_entropy_fwd(const float* logits, const int64_t* target, int64_t N, int64_t C, int mean,
                           float* loss, int32_t* bad_target, void* workspace, size_t* workspace_bytes,
                           void* stream);
int mgcn_cross_entropy_bwd(const float* logits, const int64_t* target, int64_t N, int64_t C, int mean,
                           const float* upstream, float* dlogits, void* stream);

/* The step right behind the hot path, fused (SURVEY §8 f3): self.final = nn.Linear(H, C) (gcn_model.py:73,108),
 * nn.CrossEntropyLoss (train_botnet.py:225,287) and the binary counters of optim/metrics.py:8-24
 * (train_botnet.py:296-305) as ONE forward launch that reads x [N,H] once — logits [N,C] = x w^T + b are written
 * because the caller returns them; loss[0] = sum (or mean) of the rows' NLL, fixed-order; counts5 = {TP, FP, TN, FN,
 * correct} (int64, may be NULL) — and ONE backward launch that reads x and the logits once:
 *   dl = (softmax(logits) - onehot(target)) * (1/N if mean) * upstream[0]
 *   dx = dl w  (may be NULL);   dw = dl^T x;   db = colsum(dl)      (fixed-order partials: deterministic)
 * H in {16, 32, 64, 128}, C <= 8, w [C,H] (nn.Linear.weight), b [C] or NULL.  The row NLL, the label's gradient
 * entry, labels outside [0, C) and N = 0 follow the node-level cross entropy above. */
int mgcn_head_cross_entropy_fwd(const float* x, int64_t N, int64_t H, const float* w, const float* b, int64_t C,
                                const int64_t* target, int mean, float* logits, float* loss, int64_t* counts5,
                                int32_t* bad_target, void* workspace, size_t* workspace_bytes, void* stream);
int mgcn_head_cross_entropy_bwd(const float* x, const float* logits, int64_t N, int64_t H, const float* w, int64_t C,
                                const int64_t* target, int mean, const float* upstream, float* dx, float* dw,
                                float* db, void* workspace, size_t* workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * 'max' aggregation: scatter_('max', src, index, dim_size) (common.py:54-64 — torch_scatter scatter_max with fill
 * -1e38, untouched rows set to 0) and NodeModelAdditive(aggr='max') (gcn_base_models.py:223-237), with
 * torch_scatter's gradient rule (the first entry that attains the maximum receives the gradient).
 * out[i,c] = max over the row's entries, in row order, of edge_val[k] * x[idx_k, c] (idx = perm when gather_perm:
 * primitive seam, else nbr: layer seam; edge_val in row order or NULL); arg[i,c] = edge id (perm) of the first
 * maximal entry, -1 (and out = 0) for a row without entries.  Deterministic, no atomics.
 * mgcn_segment_max: the row's first entry always wins, whatever its value.
 * mgcn_segment_max_ex: torch_scatter's fill rule — the running maximum starts at `fill` and an entry wins only if it
 * is strictly greater, so an entry <= fill never wins; a (row, column) without a winner gives out = 0, arg = -1.
 * Callers pass the fill of the call they stand for (-1e38 for common.py's scatter_('max'), -1e9 for PyG 1.3's
 * scatter_('max'), fill_value for scatter_max).  The two agree wherever some entry of the row is > fill. */
int mgcn_segment_max(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, int gather_perm,
                     const float* edge_val, float* out, int32_t* arg, void* stream);
int mgcn_segment_max_ex(const mgcn_csr_t* g, const float* x, int64_t n_in, int64_t H, int gather_perm,
                        const float* edge_val, float fill, float* out, int32_t* arg, void* stream);
/* layer seam, gt = the structure grouped by the OTHER endpoint (by source):
 * dx[j,c] = sum over row j's entries k of [arg[nbr_k, c] == perm_k] * edge_val[k] * grad[nbr_k, c] */
int mgcn_segment_max_bwd(const mgcn_csr_t* gt, const float* grad, const int32_t* arg, const float* edge_val,
                         int64_t H, float* dx, void* stream);
/* primitive seam: dsrc [n_src,H] = 0, then dsrc[arg[i,c], c] = grad[i,c] */
int mgcn_scatter_max_bwd(const int32_t* arg, const float* grad, int64_t N, int64_t H, int64_t n_src, float* dsrc,
                         void* stream);

/* out[e] = scale_src[row_e] * scale_tgt[col_e] * sum_c a[col_e,c] * b[row_e,c]   (row = edge_index[0], col =
 * edge_index[1]; scales may be NULL): the gradient of an aggregation w.r.t. a per-edge weight, used by the edge gates
 * (gcn_base_models.py:230-232, 322-369: x_j = sigmoid(...)_e * x_j before scatter_).  Deterministic.
 * _i32: the same for an int32 edge_index (bit-identical output). */
int mgcn_edge_dot(const int64_t* edge_index, int64_t E, const float* a, const float* b, int64_t H,
                  const float* scale_src, const float* scale_tgt, float* out, void* stream);
int mgcn_edge_dot_i32(const int32_t* edge_index, int64_t E, const float* a, const float* b, int64_t H,
                      const float* scale_src, const float* scale_tgt, float* out, void* stream);

/* Binary-classification counters of src/gcn_meta/optim/metrics.py:8-24 as used at train_botnet.py:296-305:
 * counts5 = {TP, FP, TN, FN, correct} (int64) with pred = argmax(logits[n,:]) (first maximal class; logits
 * float [N,C]) or the given pred int64[N] (exactly one of logits / pred is non-NULL); target int64[N].
 * One pass, integer sums (exact); the reference makes one boolean-mask pass and one host sync per counter. */
int mgcn_binary_confusion(const float* logits, const int64_t* pred, int64_t N, int64_t C,
                          const int64_t* target, int64_t* counts5, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MGCN_H_ */
