/*
 * regt_b200.h -- C-ABI of the B200-native RegT-GCN hot path (libregt_b200.so).
 *
 * The reference (raynbowy23/RegT-GCN) has no FFI layer: its boundary for this path is the
 * Python nn.Module surface.  Every entry point below therefore names the reference
 * interface whose arithmetic it replaces (file:line under the reference tree); the
 * Python binding a maintainer adds on the reference side is shown in INTEGRATION.md and
 * implemented in regt-gcn_b200/regt_b200/_lib.py + models/*.py.
 *
 * Conventions
 *  - all pointers are DEVICE pointers unless the comment says "host";
 *  - no ownership transfer and no hidden allocation: the caller passes a workspace of at
 *    least regt_workspace_bytes() bytes (256-byte aligned);
 *  - every function returns 0 on success, <0 on error; regt_last_error() returns a
 *    thread-local message for the last failure on the calling thread;
 *  - work is enqueued on `stream`; nothing synchronises the device except the
 *    regt_gcn_plan_build / regt_cheb_plan_build calls (they return counts to the host);
 *  - thread-compatible: no global state except the thread-local error string.
 */
#ifndef REGT_B200_H
#define REGT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REGT_VERSION 100 /* 0.1.0 */
#define REGT_F 8         /* the kernels' feature width, and the largest regt_args.F (the reference uses 8, run.py:116) */

/* precision of the H x H contractions */
#define REGT_PREC_FP32 0  /* FFMA, fp32 everywhere (parity mode, all shapes)            */
#define REGT_PREC_TF32X3 1 /* tcgen05 kind::tf32, 3-pass split: fp32-equivalent accuracy  */
#define REGT_PREC_BF16 2  /* tcgen05 kind::f16 bf16 operands, fp32 accumulate: the fused cell at hidden 64
                             (not the bare TGCN cell), the single-pass bf16 GEMMs at every other hidden % 32 == 0 */

typedef void* regt_stream_t; /* cudaStream_t */

/* ---- K1: static-graph plan ---------------------------------------------------------- */
/* CSR by destination of the normalised operators, built once per static graph.
 * Canonical order (bit-exact contract): PyG's post-normalisation edge list, stable-sorted
 * by destination; duplicates kept. */
typedef struct regt_graph_plan {
  int32_t N;        /* nodes */
  int32_t nnz_gcn;  /* E' + N  (E' = non-loop edges of edge_index)                       */
  int32_t nnz_cheb; /* non-loop edges of all regional lists                              */
  int32_t nseg;     /* number of (node, region) segments with at least one in-edge       */
  int32_t R;        /* number of regional edge lists (1 for A3TGCN)                      */
  int32_t _pad;
  const int32_t* g_rowptr; /* [N+1]                                                      */
  const int32_t* g_col;    /* [nnz_gcn] sources                                          */
  const float* g_val;      /* [nnz_gcn] D~^-1/2 (A+I) D~^-1/2 entries (gcn_norm)          */
  const int32_t* c_rowptr; /* [N+1]                                                      */
  const int32_t* c_col;    /* [nnz_cheb]                                                 */
  const float* c_val;      /* [nnz_cheb] -D^-1/2 A D^-1/2 entries (ChebConv, K=2, sym)    */
  const int32_t* c_reg;    /* [nnz_cheb] regional list id of every entry                  */
  const int32_t* seg_ptr;  /* [N+1]   segments of node n are seg_ptr[n]..seg_ptr[n+1]     */
  const int32_t* seg_eptr; /* [nseg+1] entry range of each segment inside the cheb CSR    */
  const int32_t* seg_reg;  /* [nseg]                                                     */
  const int32_t* seg_node; /* [nseg]                                                     */
  const int32_t* rseg_ptr; /* [R+1]   segments grouped by region: rseg_list[rseg_ptr[r]..]    */
  const int32_t* rseg_list;/* [nseg]  segment ids, ascending inside a region                  */
} regt_graph_plan;

/* replaces torch_geometric gcn_norm + scatter index of GCNConv.propagate, which the
 * reference re-runs 3*T times per sample (models/utils.py:169,175,181; cached=False :81).
 * edge_index int64 [2,E] (row 0 = source, row 1 = target), edge_weight f32 [E] or NULL.
 * Outputs: rowptr [N+1], col/val [E+N] (upper bound), eid [E+N] = position of every CSR
 * entry in PyG's post-normalisation edge list (for tests).  *nnz_out (host) = E'+N.   */
size_t regt_plan_workspace_bytes(int64_t num_nodes, int64_t num_edges);
int regt_gcn_plan_build(const int64_t* edge_index, const float* edge_weight, int64_t E, int64_t N,
                        int32_t* rowptr, int32_t* col, float* val, int32_t* eid, int32_t* nnz_out /*host*/,
                        void* workspace, size_t workspace_bytes, regt_stream_t stream);

/* replaces torch_geometric get_laplacian('sym') + Chebyshev rescale inside ChebConv.forward,
 * which the reference re-runs R*T times per sample (models/RegionalTemporalGCN.py:136-140,
 * models/TemporalGCN.py:88).  The R regional lists are passed concatenated:
 * edge_index int64 [2,E_tot], edge_weight f32 [E_tot] or NULL, list_ptr (host) int64 [R+1].
 * Each list is normalised on its own (source degree inside that list).
 * Outputs (upper bounds): rowptr [N+1], col/val/reg/eid [E_tot], seg_ptr [N+1],
 * seg_eptr [E_tot+1], seg_reg/seg_node/rseg_list [E_tot], rseg_ptr [R+1],
 * region_of [N] (-1 untouched, -2 in >1 list).  counts_out (host) int32[2] = {nnz, nseg}. */
int regt_cheb_plan_build(const int64_t* edge_index, const float* edge_weight, const int64_t* list_ptr /*host*/,
                         int32_t R, int64_t E_tot, int64_t N, int32_t* rowptr, int32_t* col, float* val,
                         int32_t* reg, int32_t* eid, int32_t* seg_ptr, int32_t* seg_eptr, int32_t* seg_reg,
                         int32_t* seg_node, int32_t* rseg_ptr, int32_t* rseg_list, int32_t* region_of,
                         int32_t* counts_out /*host*/, void* workspace, size_t workspace_bytes,
                         regt_stream_t stream);

/* ---- stand-alone F-wide SpMM (BASELINE metric "SpMM HBM GB/s") ----------------------- */
/* y[b,n,:] = sum_{e in row n} val[e] * x[b,col[e],:]  for rows of `width` floats
 * (width = F*T = 96 for the x[B,N,F,T] layout of load_dataset.py:456; width % 4 == 0).
 * Replaces GCNConv.propagate's index_select/mul/scatter_add (models/utils.py:169).      */
int regt_spmm_f8(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y,
                 int32_t B, int32_t N, int32_t width, regt_stream_t stream);
/* Plan-time row partition for the staged SpMM kernel (once per static graph, like gcn_norm's plan: the reference
 * re-derives the same index structure on every GCNConv call, models/utils.py:169).  The kernel stages a block of
 * consecutive node rows in shared memory and gathers from there; regt_spmm_partition cuts the rows into blocks that
 * fit, at the positions the fewest edges cross (region borders when node ids are ordered by region), so that nearly
 * all neighbour reads stay on chip.  blk_ptr: device int32[regt_spmm_partition_capacity(N, width)] (0: rows too wide
 * for the staged kernel), receives nblk+1 row offsets; nblk_out: host.  Synchronises the stream (copies the CSR back).
 * regt_spmm_f8_blocked computes exactly what regt_spmm_f8 does (same order of additions: bit-identical).           */
int32_t regt_spmm_partition_capacity(int32_t N, int32_t width);
int regt_spmm_partition(const int32_t* rowptr, const int32_t* col, int32_t N, int32_t width, int32_t* blk_ptr,
                        int32_t* nblk_out /*host*/, regt_stream_t stream);
int regt_spmm_f8_blocked(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y,
                         int32_t B, int32_t N, int32_t width, const int32_t* blk_ptr, int32_t nblk,
                         regt_stream_t stream);

/* ---- K4: regional gather / scatter of node rows -------------------------------------- */
/* The reference has no node subsets (a region is an edge list over global ids,
 * models/RegionalTemporalGCN.py:136-140; the slices of load_dataset.py:458-467 are computed and
 * discarded); the region-sharded multi-GPU path needs them: a rank's input is its owned rows
 * followed by the 1-hop halo rows, its outputs are scattered back into global node order.
 *   gather : dst[b][i][:] = src[b][idx[i]][:]   src [B,n_src,width], dst [B,n_idx,width]
 *   scatter: dst[b][idx[i]][:] = src[b][i][:]   src [B,n_idx,width], dst [B,n_dst,width]
 * idx int64 [n_idx] (device), rows of `width` floats.                                     */
int regt_gather_rows(const float* src, const int64_t* idx, float* dst, int32_t B, int32_t n_src, int32_t n_idx,
                     int32_t width, regt_stream_t stream);
int regt_scatter_rows(const float* src, const int64_t* idx, float* dst, int32_t B, int32_t n_idx, int32_t n_dst,
                      int32_t width, regt_stream_t stream);

/* ---- the cell + head ---------------------------------------------------------------- */
typedef struct regt_params {            /* reference state_dict layouts (SURVEY 8(b))      */
  float* attention;                     /* tgnn._attention [T]                             */
  float* conv_w[3];                     /* tgnn._base_tgcn.conv_{z,r,h}.lin.weight [H,F]    */
  float* conv_b[3];                     /* tgnn._base_tgcn.conv_{z,r,h}.bias [H]            */
  float* lin_w[3];                      /* tgnn._base_tgcn.linear_{z,r,h}.weight [H,2H]     */
  float* lin_b[3];                      /* tgnn._base_tgcn.linear_{z,r,h}.bias [H]          */
  float* cheb_w0;                       /* tgnn.conv.lins.0.weight [H,F]                   */
  float* cheb_w1;                       /* tgnn.conv.lins.1.weight [H,F]                   */
  float* cheb_b;                        /* tgnn.conv.bias [H]                              */
  float* comb_w;                        /* tgnn.linear.weight [H,R*H]   (regional only)     */
  float* comb_b;                        /* tgnn.linear.bias [H]         (regional only)     */
  float* head_w1;                       /* linear1.weight [128,H]                          */
  float* head_b1;                       /* linear1.bias [128]                              */
  float* head_w2;                       /* linear2.weight [O,128]                          */
  float* head_b2;                       /* linear2.bias [O]                                */
} regt_params;

#define REGT_MODE_REGIONAL 1 /* RegionalA3TGCN: R ChebConvs -> Linear(R*H,H) -> leaky_relu  */
#define REGT_MODE_A3TGCN 0   /* A3TGCN: h = ChebConv(X_t) on the full graph                */
#define REGT_MODE_TGCN 2     /* bare TGCN cell: h supplied by the caller (or zeros)         */

typedef struct regt_args {
  int32_t B, N, T, H, O;  /* x is [B,N,F,T]; T = periods; O = output_dim                  */
  int32_t mode;           /* REGT_MODE_*                                                  */
  int32_t precision;      /* REGT_PREC_*                                                  */
  int32_t accumulate;     /* backward: 0 overwrite param grads, 1 add into them           */
  int32_t fuse_head;      /* 1 (needs y): head_forward also runs the head's backward (d_out,  */
                          /*    gradient wrt out_hidden, weight-gradient partials) in the same */
                          /*    kernel; head_backward then only reduces the partials           */
  int32_t x_rows;         /* region shards: node rows per snapshot of x (>= N; 0 means N).     */
                          /*    Rows [0,N) are the nodes this call owns (outputs are written   */
                          /*    for them); rows [N,x_rows) are halo inputs that only the plan's */
                          /*    column indices address (1-hop neighbours owned by other ranks). */
  int32_t loss_nodes;     /* region shards: node count of the loss mean (0 means N), so that   */
                          /*    the per-rank losses and gradients ADD to the full-graph ones    */
  int32_t inference;      /* 1: forward only, as under torch.no_grad() at run.py:208-216 / predict.py:151-172:    */
                          /*    the fused kernels save no activations (the workspace shrinks accordingly) and     */
                          /*    regt_head_backward / regt_cell_backward must not follow                           */
  regt_graph_plan plan;
  const float* x;         /* [B,x_rows,F,T] f32, T innermost (load_dataset.py:456); 16-byte aligned at F = REGT_F,  */
                          /*    4-byte aligned suffices below (x is then read with scalar loads only)             */
  const float* y;         /* [B,N,O] or NULL: if set head_forward also writes loss, d_out  */
  const float* h_ext;     /* REGT_MODE_TGCN: [B,N,T,H] state or NULL (= zeros)            */
  regt_params p;          /* parameters                                                   */
  regt_params g;          /* parameter gradients (same layouts; any may be NULL)          */
  float* out_hidden;      /* [B,N,H]  cell output (pre-ReLU), models/RegionalTemporalGCN.py:34 */
  float* out;             /* [B,N,O]                                                      */
  float* loss;            /* [1]  sum_b mean_{n,o} l(out-y)  (run.py:180; l = loss_kind); with loss_masked the mean of  */
                          /*    snapshot b runs over its valid targets only: sum_b [c_b > 0] sum_{n,o} m l / c_b        */
  float* d_out;           /* [B,N,O]  gradient of loss wrt out (in/out); with loss_masked m l' / c_b (0 where c_b = 0)  */
  float* d_hidden;        /* [B,N,H]  extra gradient flowing into out_hidden, or NULL     */
  float* d_h_ext;         /* REGT_MODE_TGCN: [B,N,T,H] gradient wrt h_ext, or NULL        */
  void* workspace;        /* regt_workspace_bytes(args) bytes, preserved fwd -> bwd       */
  size_t workspace_bytes;
  regt_stream_t stream;
  int32_t F;              /* features per node of x, 1..REGT_F; 0 means REGT_F.  x, conv_w, cheb_w0 / cheb_w1 and    */
                          /*    their gradients have this width; the kernels work at REGT_F with the features and   */
                          /*    weight columns F..REGT_F-1 written as zeros, so the result is that of the REGT_F-wide */
                          /*    model on zero-padded x and weights                                                  */
  int32_t loss_kind;      /* REGT_LOSS_*: l = (out-y)^2, l' = 2(out-y) (MSE, 0) or l = |out-y|, l' = sign(out-y) (MAE)  */
  int32_t loss_masked;    /* 1: target y[b,n,o] is missing when it equals loss_null or is NaN; m = 0 there, else 1.     */
                          /*    0: no mask (a NaN in y propagates).  The kernels run their unmasked MSE code unchanged  */
                          /*    when loss_kind = 0 and loss_masked = 0                                                 */
  float loss_null;        /* the value that marks a missing target (NaN: only NaNs are missing)                        */
  const float* loss_count;/* [B] valid count c_b of each snapshot over ALL nodes of the graph (region shards: the full   */
                          /*    graph's counts), or NULL: counted over rows [0,N) of y on the device                   */
  int32_t head_only;      /* 1: the call runs the head (and loss) on a given out_hidden, with no cell: the workspace holds  */
                          /*    no cell planes, regt_cell_* refuse the args, the head never runs k_head_tc, and the         */
                          /*    gradient wrt out_hidden, G [B*N][H] row major, is left at the START of the workspace by     */
                          /*    regt_head_backward (what regt_combine_backward reads).  0: the full step, as before        */
} regt_args;

#define REGT_LOSS_MSE 0
#define REGT_LOSS_MAE 1

size_t regt_workspace_bytes(const regt_args* a);

/* replaces RegionalA3TGCN.forward (models/RegionalTemporalGCN.py:114-149) /
 * A3TGCN.forward (models/TemporalGCN.py:75-91) / TGCN.forward (models/utils.py:190-203):
 * weight collapse, F-wide SpMM, regional combine, GRU gates, period attention.
 * Writes out_hidden and the saved activations inside the workspace.                    */
int regt_cell_forward(const regt_args* a);
/* replaces the head of RegionalTemporalGCN.forward / TemporalGCN.forward
 * (models/RegionalTemporalGCN.py:35-38, models/TemporalGCN.py:28-31) and, when y is
 * given, the loss of the call site (run.py:180).                                        */
int regt_head_forward(const regt_args* a);
/* autograd of the head (run.py:190): consumes d_out, writes g.head_* and the gradient
 * wrt out_hidden (kept in the workspace for regt_cell_backward).  With fuse_head=1 in precision
 * bf16 the head ran its backward inside regt_head_forward and left per-CTA partials; their sum
 * (g.head_*, loss) is then finalised by the regt_cell_backward that must follow, beside the cell
 * kernel on a second stream.                                                             */
int regt_head_backward(const regt_args* a);
/* autograd of the cell (run.py:190): all parameter gradients of the cell.  The gradient wrt x
 * is not part of this call (x is data in the reference's loop: batch.x never requires grad);
 * regt_cell_backward_x below computes it from what this call leaves in the workspace.    */
int regt_cell_backward(const regt_args* a);

/* ---- gradient wrt x (csrc/input_grad.cu) ----------------------------------------------
 * What autograd gives PyG's modules for an x that requires grad (saliency, input perturbation,
 * an upstream layer feeding models.utils.TGCN).  Per row (b, n, t) the gate-gradient plane
 * D = [Dz | Dr | Dc | Dpre] of the cell backward is contracted with the collapsed weights into
 *   dS = Dzr (A_zr W_zr) + Dc (A_c W_c),  dXd = Dpre M0,  dU_seg = Dpre M1[r_seg]  (F wide each),
 * then  dx = dXd + A_hat^T dS + sum_r C_r^T dU  (the graphs are directed: neither transpose
 * equals its operator).  The transposed operator is one CSR by input node j over the stacked
 * source rows [dXd (N) | dS (N) | dU (nseg)] of a snapshot; row j holds, in this fixed order, the
 * identity entry (dXd row j, weight 1), then the A_hat entries with g_col = j, then the regional
 * entries with c_col = j, each group in canonical CSR order: sums are deterministic.          */
typedef struct regt_xgrad_plan {
  int32_t N;              /* nodes                                                          */
  int32_t nnz;            /* N + nnz_gcn + nnz_cheb                                         */
  int32_t n_src;          /* 2 N + nseg: stacked source rows of one snapshot                */
  int32_t _pad;
  const int32_t* rowptr;  /* [N+1]                                                          */
  const int32_t* col;     /* [nnz] stacked source row                                       */
  const float* val;       /* [nnz] 1 (identity), g_val or c_val of the entry                */
} regt_xgrad_plan;

/* Built once per static graph from a regt_graph_plan (stable counting sort by column, on the
 * device; all sizes come from the plan, so it does not synchronise).  Outputs: rowptr [N+1],
 * col / val [N + nnz_gcn + nnz_cheb].                                                         */
size_t regt_xgrad_plan_workspace_bytes(const regt_graph_plan* p);
int regt_xgrad_plan_build(const regt_graph_plan* p, int32_t* rowptr, int32_t* col, float* val, void* workspace,
                          size_t workspace_bytes, regt_stream_t stream);
/* d_x [B,N,F,T] f32 (F = regt_args.F; overwritten) = gradient wrt x of the loss whose gradients the preceding
 * regt_cell_backward (same args, same workspace) consumed.  Reads the workspace, allocates nothing:
 * scratch is at least regt_cell_backward_x_scratch_bytes(a, xp) bytes (256-byte aligned).
 * Refused: precision bf16 (its kernels keep no D plane), region shards (x_rows != N: halo rows
 * belong to other ranks), inference = 1 (no backward ran).                                    */
size_t regt_cell_backward_x_scratch_bytes(const regt_args* a, const regt_xgrad_plan* xp);
int regt_cell_backward_x(const regt_args* a, const regt_xgrad_plan* xp, float* d_x, void* scratch, size_t scratch_bytes);

/* ---- exchange step over NVLink peer memory (csrc/peer.cu) ------------------------------
 * SURVEY 8e: one sum all-reduce of the flat shared-weight gradient buffer per step.  The
 * reference has no distributed path; these entry points replace what a DistributedDataParallel
 * wrapper around run.py:190 would do with NCCL.  A rank allocates ONE communication region
 * [flags | data | scratch], the others map it through CUDA IPC; the wgrad kernels write
 * straight into `data`; regt_peer_allreduce_f32 is a single kernel (per-block flag barrier,
 * peer reads in rank order -> bit-identical sums on every rank, copy back), capturable in a
 * CUDA graph.  Explicit allocation: a peer-mappable region must be a whole cudaMalloc block. */
size_t regt_comm_region_bytes(int64_t n_floats);
size_t regt_comm_data_offset(void);
int regt_comm_alloc(size_t bytes, void** ptr);
int regt_comm_free(void* ptr);
int regt_comm_export(void* ptr, unsigned char* handle64 /*host, 64 bytes*/);
int regt_comm_import(const unsigned char* handle64 /*host*/, void** peer_ptr);
int regt_comm_unimport(void* peer_ptr);
/* last_in (optional, device): added to this rank's element n_floats - 4 (the loss slot) before the sum;
 * last_out (optional, device): receives the reduced loss slot, which is then cleared.  Both need n_floats <= 2^18. */
int regt_peer_allreduce_f32(void* const* regions /*host array [world]*/, int32_t rank, int32_t world, int64_t n_floats,
                            const float* last_in, float* last_out, regt_stream_t stream);
int64_t regt_peer_push_max_floats(void);
int regt_comm_error(void* region);

/* ---- callers on either side of the path, on the device (csrc/loop.cu; SURVEY 8f.1 / 8f.2) ----
 * regt_window_gather: load_dataset.py:451-457 + run.py:172 -- x[b,n,f,t] = node_data[n,f,starts[b]+t],
 *   y[b,n,o] = node_data[n,target_f,starts[b]+T_in+o]; node_data [N,F,T_total] stays resident.
 * regt_rmsprop_step: run.py:145,194 -- torch.optim.RMSprop (no momentum, not centred) over flat buffers.
 * regt_eval_metrics: predict.py:142-194 -- sums[b] = { sum|y-out|, sum (y-out)^2, percentile q of y_b (numpy
 *   'linear'), sum|y-out| / percentile } as doubles; the host combines them (regt_b200/loop.py). */
int regt_window_gather(const float* node_data, const int64_t* starts, int32_t B, int32_t N, int32_t F, int64_t T_total,
                       int32_t T_in, int32_t T_out, int32_t target_f, float* x, float* y, regt_stream_t stream);
int regt_rmsprop_step(float* params, const float* grads, float* square_avg, int64_t n, float lr, float alpha, float eps,
                      float weight_decay, regt_stream_t stream);
int regt_eval_metrics(const float* out, const float* y, int32_t B, int64_t n_per_snapshot, double q, double* sums,
                      regt_stream_t stream);
/* regt_eval_metrics over the valid targets only (y != null_value and not NaN; null_value NaN: only NaNs are missing):
 *   sums[b] = { valid count c_b, sum m|y-out|, sum m (y-out)^2, percentile q of the valid y_b, sum m|y-out| / percentile }
 * as doubles [B][5]; a snapshot with c_b = 0 gives {0, 0, 0, NaN, NaN}.                                                   */
int regt_eval_metrics_masked(const float* out, const float* y, int32_t B, int64_t n_per_snapshot, double q, float null_value,
                             double* sums, regt_stream_t stream);

/* ---- time steps shared across sliding windows (csrc/combine.cu; regt_b200/loop.py share_periods) --------------------
 * The cell output of a period depends on that period's input alone (the hidden state is not carried across periods), so
 * the cell output H'(tau) of time step tau is the same in every window that contains tau.  A pass over C consecutive
 * windows runs the cell once per time step, S = C + T - 1 steps (regt_cell_forward at T = 1 over S "snapshots"), then
 *   regt_combine_forward:  out_hidden[w] = sum_{t<T} p_t H'[w+t]        (w < C; summed in period order)
 *   regt_combine_backward: Gs[tau]      = sum_{t<T, 0 <= tau-t < C} p_t G[tau-t]     (tau < S; in period order)
 *                          dprobs_t     = sum_w <G[w], H'[w+t]>  (fp64 partials, summed in a fixed order)
 *                          attention_grad[t] += p_t (dprobs_t - sum_s p_s dprobs_s)     (when attention_grad is set)
 * p = softmax(attention [T]), computed as the cell kernels compute it.  Hs / Gs [S][width], out_hidden / G [C][width],
 * width = N*H (a multiple of 4; 16-byte aligned rows).  Each element of Hs and G is read once when width fills the device;
 * a narrower pass is split into chunks of windows (steps) that re-read T - 1 rows each.  Gs is the gradient wrt the
 * step cell's out_hidden (regt_args.d_hidden of its regt_head_backward with d_out = NULL).
 * scratch: at least regt_combine_scratch_bytes(T) bytes (backward only; 8-byte aligned).                               */
size_t regt_combine_scratch_bytes(int32_t T);
int regt_combine_forward(const float* attention, const float* Hs, int32_t S, int32_t C, int32_t T, int64_t width, float* out_hidden,
                         regt_stream_t stream);
int regt_combine_backward(const float* attention, const float* Hs, const float* G, int32_t S, int32_t C, int32_t T, int64_t width,
                          float* Gs, float* attention_grad, void* scratch, size_t scratch_bytes, regt_stream_t stream);

int regt_version(void);
const char* regt_last_error(void);
/* number of kernel launches issued by this library on the calling thread since the last
 * call with reset != 0 (bench.py's "gpu_launches").                                     */
int64_t regt_launch_count(int reset);

/* per-kernel timing for bench.py's roofline: while enabled, every kernel launch of this
 * library is followed by a cudaEventRecord on the launching stream.  regt_profile_begin()
 * re-arms the interval origin; regt_profile_read() synchronises and returns, for each launch,
 * the time since the previous mark ('\n'-separated names; ms[i]).  Not for use under graph
 * capture.  No reference counterpart (the reference has no profiling, SURVEY section 5).     */
int regt_profile(int enable, regt_stream_t stream);
int regt_profile_begin(regt_stream_t stream);
int regt_profile_read(char* names, size_t names_len, float* ms, int max_n);

/* ---- TEST HOOKS ------------------------------------------------------------------------------------------------
 * Not part of the reference-facing boundary: no reference call site maps to these.  They expose the internal
 * tensor-core building blocks (3xTF32 and bf16 GEMMs of gemm_tma.cu, the hand-built UMMA operand layouts of
 * tc_common.cuh) to tests/test_gpu_gemm.py and tests/test_gpu_umma.py so that each is pinned against an fp64 matmul on
 * its own.  Integrators do not bind them.
 *   gemm_nt_tma:  C[M][N]   = A[M][K] . Bt[N][K]^T                    (scratch: 2 * ceil128(N) * ceil32(K) floats)
 *   gemm_tn_tma:  Cp[z]     = sum over the rows of split z of A[r][:K]^T . B[r][:N]      (+ a second, 32-wide operand B2)
 *   gemm_nt_bf16, gemm_tn_bf16: the same two products with both operands rounded to bf16 once (single-pass kind::f16,
 *                 fp32 accumulate), same arguments; gemm_nt_bf16 needs ceil128(N) * ceil64(K) / 2 floats of scratch
 *   gemm_tn_multi: the four-gate-block form of the cell backward, A = D [M][4H] (gemm_tn_multi_bf16: its bf16 form)
 *   gemm_kt: the same contraction over transposed tiles A^T [ntile][4H][128], B^T [ntile][H][128], F^T [ntile][32][128]
 *            (what the fused cell backward of cell_f.cu writes); H = 128 or 64
 *   umma_selftest: one 128 x N x K MMA on operand tiles written by CUDA-core threads (fmt 1 = bf16, 2 = tf32)
 *   tc_split: how the bf16 kernels of cell_tc.cu / head_tc.cu split B*N rows over T periods on this device, written to
 *             out[7] = {128-row tiles nqt, periods per item tp, period chunks ntc = T / tp, items = nqt * ntc,
 *             forward grid, backward grid, k_head_tc grid} (tests/test_gpu_bf16_edges.py states its preconditions so)
 *   route: which cell and head kernels the entry points run for these arguments (no CUDA call, no workspace needed),
 *          out[4] = {cell: 0 fp32, 1 unfused tf32x3, 2 fused tf32x3, 3 fused bf16, 4 GEMM-by-GEMM bf16, 5 none (head_only);
 *          head: 0 row kernels k_head_fwd / k_head_bwd,
 *          1 k_head_fused, 2 tf32x3 head, 3 k_head_tc; G written as tiles; bf16 forward leaves out_hidden partials}   */
int regt_debug_gemm_nt_tma(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc, int64_t M,
                           int32_t N, int32_t K, float* scratch, regt_stream_t stream);
int regt_debug_gemm_tn_tma(const float* A, int64_t lda, const float* B, int64_t ldb, float* Cp, int64_t M, int32_t K,
                           int32_t N, int32_t splits, const float* B2, int64_t ldb2, float* Cp2, regt_stream_t stream);
int regt_debug_gemm_nt_bf16(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc, int64_t M,
                            int32_t N, int32_t K, float* scratch, regt_stream_t stream);
int regt_debug_gemm_tn_bf16(const float* A, int64_t lda, const float* B, int64_t ldb, float* Cp, int64_t M, int32_t K,
                            int32_t N, int32_t splits, const float* B2, int64_t ldb2, float* Cp2, regt_stream_t stream);
int regt_debug_gemm_tn_multi(const float* A, int64_t lda, int64_t M, int32_t H, const float* B0, const float* B1,
                             float* C0, float* C1, int32_t splits, const float* B2, float* C2, regt_stream_t stream);
int regt_debug_gemm_tn_multi_bf16(const float* A, int64_t lda, int64_t M, int32_t H, const float* B0, const float* B1,
                                  float* C0, float* C1, int32_t splits, const float* B2, float* C2, regt_stream_t stream);
int regt_debug_gemm_kt(const float* AT, int64_t ntile, int32_t H, const float* B0T, const float* B1T, const float* FT,
                       float* C0, float* C1, float* C2, int32_t splits, regt_stream_t stream);
int regt_debug_spmm_partition_host(const int32_t* rowptr, const int32_t* col, int32_t N, int32_t width, int32_t* blk_ptr,
                                   int32_t* nblk_out, int32_t* cap_out);   /* regt_spmm_partition's algorithm on HOST arrays; cap_out = {rows, edges} a block may hold */
int regt_debug_f_timestamps(long long* out);   /* phase clocks of the fused 3xTF32 cell kernels (REGT_F_DEBUG), [3][16][12]: forward epilogue, backward epilogue, forward MMA warp */
int regt_debug_umma_selftest(int fmt, int variant, const float* A, const float* B, float* D, int N, int K,
                             regt_stream_t stream);
int regt_debug_tc_split(int32_t B, int32_t N, int32_t T, int32_t* out);
int regt_debug_route(const regt_args* args, int32_t* out);

#ifdef __cplusplus
}
#endif
#endif /* REGT_B200_H */
