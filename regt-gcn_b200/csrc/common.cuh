// Shared helpers for libregt_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "regt_b200.h"

namespace regt {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void prof_mark(const char* name, cudaStream_t st);
// fork: returns a library-owned side stream that waits for everything enqueued on `main` so far (or
// nullptr: run serially); join: `main` waits for everything enqueued on the side stream
cudaStream_t fork_side(cudaStream_t main);
int join_side(cudaStream_t main);

#define REGT_CHECK(cond, ...)         \
  do {                                \
    if (!(cond)) {                    \
      regt::set_error(__VA_ARGS__);   \
      return -1;                      \
    }                                 \
  } while (0)

#define REGT_CUDA(expr)                                                                  \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      regt::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -2;                                                                         \
    }                                                                                    \
  } while (0)

#define REGT_LAUNCH_CHECK()                                                              \
  do {                                                                                   \
    regt::count_launch();                                                                \
    cudaError_t _e = cudaGetLastError();                                                 \
    if (_e != cudaSuccess) {                                                             \
      regt::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -3;                                                                         \
    }                                                                                    \
  } while (0)

// like REGT_LAUNCH_CHECK, and (when regt_profile(1) is active) records a CUDA event on the
// launching stream so that consecutive marks bracket every kernel of the step
#define REGT_LAUNCHED(name, st)       \
  do {                                \
    REGT_LAUNCH_CHECK();              \
    regt::prof_mark(name, st);        \
  } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// bump allocator over the caller's workspace
struct Carver {
  char* base;
  size_t off;
  explicit Carver(void* p) : base((char*)p), off(0) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* r = base ? (T*)(base + off) : (T*)nullptr;
    off += n * sizeof(T);
    return r;
  }
};

__device__ __forceinline__ float sigmoidf_(float v) { return 1.0f / (1.0f + expf(-v)); }

// softmax over the T learned period-attention scalars (models/RegionalTemporalGCN.py:134), one thread: what k_prep writes
// to Layout::probs and what the period-sharing combine kernels (combine.cu) weight the time steps with
__device__ __forceinline__ void attention_softmax(const float* att, int T, float* probs) {
  float mx = -INFINITY;
  for (int t = 0; t < T; ++t) mx = fmaxf(mx, att[t]);
  double den = 0.0;
  for (int t = 0; t < T; ++t) den += exp((double)att[t] - mx);
  for (int t = 0; t < T; ++t) probs[t] = (float)(exp((double)att[t] - mx) / den);
}

// offset of G[q][n] (gradient wrt out_hidden): row major, or the [qt][H/4][128][4] tiles the fused cell backwards read
__device__ __forceinline__ size_t g_off(long long q, int n, int H, int tiled) {
  return tiled ? ((((size_t)(q >> 7) * (H >> 2) + (n >> 2)) * 128 + (size_t)(q & 127)) * 4 + (n & 3)) : ((size_t)q * H + n);
}

// ---- loss of the head kernels (regt_args.loss_kind / loss_masked / loss_null / loss_count) ---------------------------
// Every head kernel is instantiated twice: LX = false is the unmasked MSE of run.py:180 with its arithmetic unchanged;
// LX = true reads the loss kind and the mask from a LossX (uniform branches) and scales each row by its snapshot's
// 1 / valid count.  Its loss is accumulated in two sums: `lu` for rows whose scale equals the unmasked one (multiplied
// once at the end, as the unmasked kernel does) and `ls` for the others (scaled per element), so a mask that finds no
// missing target gives the unmasked result bit for bit.
struct LossX {
  int mae;             // 0: (out - y)^2, 1: |out - y|
  int masked;          // 1: a target equal to null_v, or NaN, is missing
  float null_v;
  const float* inv_c;  // [B] 1 / valid count of each snapshot (0 when it has none), or NULL: the unmasked scale
  int N;               // rows per snapshot of this call: row q belongs to snapshot q / N
};
__device__ __forceinline__ float lossx_inv(const LossX& L, long long q, float scale) {
  return L.inv_c ? __ldg(L.inv_c + q / L.N) : scale;
}
// one target: adds its loss to lu or ls and returns d_out = m * l'(out - y) * inv
__device__ __forceinline__ float lossx_elem(const LossX& L, float v, float yv, float inv, float scale, float& lu, float& ls) {
  const bool keep = !L.masked || (yv == yv && yv != L.null_v);
  const float diff = keep ? v - yv : 0.f;
  if (L.mae) {
    const float l = fabsf(diff);
    if (inv == scale) lu += l;
    else ls = fmaf(l, inv, ls);
    return (diff > 0.f ? 1.f : diff < 0.f ? -1.f : diff) * inv;   // sign, 0 at 0 (torch's abs backward); NaN stays NaN
  }
  if (inv == scale) lu = fmaf(diff, diff, lu);
  else ls = fmaf(diff * diff, inv, ls);
  return 2.0f * diff * inv;
}
inline bool loss_ext(const regt_args* a) { return a->y && (a->loss_kind != REGT_LOSS_MSE || a->loss_masked); }

// multiprocessor count of the current device (148 when it cannot be read)
inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

// ---- which cell and head kernels a call runs (route_of, api.cu) ----------------------
// cell.cu, cell_g.cu, cell_f.cu, cell_tc.cu, and cell_g.cu on the single-pass bf16 GEMMs (every hidden % 32 == 0 width)
// None: a head-only call (regt_args.head_only), which runs no cell
enum class CellPath { Fp32, Tf32x3Unfused, Tf32x3Fused, Bf16, Bf16Gemm, None };
enum class HeadPath { Rows, FusedFfma, Tf32x3, Bf16 };             // k_head_fwd / k_head_bwd, k_head_fused, head_f.cu, k_head_tc
struct Route {
  CellPath cell;
  HeadPath head;
  bool g_tiled;        // G is written as tiles (g_off): the fused tf32x3 and bf16 cell backwards read it so
  bool hid_partials;   // the bf16 forward leaves per-chunk partials of out_hidden and the head sums them (no k_hid_reduce)
};
// head_only: cell None, never k_head_tc, row-major G, no out_hidden partials.
// reads REGT_UNFUSED ("1": the GEMM-by-GEMM tf32x3 cell of cell_g.cu wherever the fused one would run); no CUDA calls
Route route_of(const regt_args* a);
// the shapes each implementation is built for, with no knowledge of the other paths
bool cell_f_fits(const regt_args* a);   // fused tf32x3 cell: hidden 64 / 128, not the bare TGCN cell, <= 64 periods
bool cell_tc_fits(const regt_args* a);  // fused bf16 cell: hidden 64, not the bare TGCN cell
bool head_fused_fits(int H, int O);     // k_head_fused: hidden 32 / 64, <= 64 outputs, within a block's shared memory
bool head_tc_fits(int H, int O);        // k_head_tc: hidden 64, <= 16 outputs
bool head_f_fits(int O);                // k_hf_mid: <= 16 outputs

// ---- workspace layout shared by forward / backward (cell.cu, head.cu, api.cu) -------
struct Layout {
  Route route;   // the kernels of this call: the layout below and every launcher follow it
  // collapsed weights (rebuilt every forward: parameters change between steps)
  float* Wzr;    // [F+H][2H]   rows 0..F-1: (A_g W_g)^T, rows F..: B_g^T ; cols 0..H-1 z, H..2H-1 r
  float* Wc;     // [F+H][H]
  float* czr;    // [2H]        A_g b_g + linear_g.bias
  float* cc;     // [H]
  float* M0t;    // [F][H]      (sum_r L_r W0)^T          (A3TGCN: W0^T)
  float* M1t;    // [R][F][H]   (L_r W1)^T                (A3TGCN: W1^T)
  float* c0;     // [H]         (sum_r L_r) b + b_lin     (A3TGCN: b)
  float* Lsum;   // [H][H]      sum_r L_r                 (regional only)
  float* probs;  // [T]
  // F-wide features
  float* S;      // [B*N][F][T]      A_hat X
  float* U;      // [B][nseg][F][T]  L_hat_r X per (node, region) segment
  // saved planes, row = (b*N+n)*T + t
  float* h;      // [rows][H]
  float* Z;
  float* Rg;
  float* Hc;     // candidate H~
  float* hR;     // h * R
  float* Hn;     // H' (cell output per period)
  // head
  float* a1;     // [B*N][128]  relu(linear1(relu(hid)))
  float* G;      // [B*N][H]    gradient wrt out_hidden (head_only: row major, at the start of the workspace)
  float* d_a1;   // [B*N][128]
  // backward planes
  float* D;      // [rows][4H]  d_pre_z | d_pre_r | d_pre_h | d_hpre
  float* Feat;   // [rows][32]  S_t | X_t | 1 | 0  (tf32x3: B operand of the F-wide weight-gradient GEMM)
  // tensor-core head (head_f.cu, precision tf32x3)
  float* hf_rh;      // [BN][H]   relu(out_hidden) forward, then the unmasked gradient wrt out_hidden backward
  float* hf_do32;    // [BN][32]  d_out | 1 (column 16): feature-plane operand of the head's weight-gradient contractions
  float* hf_split;   // hi | lo images of the weight operand of the head GEMMs
  float* hf_loss;    // per-block loss partials
  size_t hf_loss_floats;
  float* FeatT;  // fused tf32x3 cell: transposed feature tiles [T*nqt][32][128] (cell_f.cu)
  float* bsplit; // GEMM-by-GEMM cell: hi | lo (tf32x3) or bf16 image of the weight operand of the current gate GEMM (gemm_tma.cu)
  // collapsed-weight gradients
  float* dB;     // [3][H][H]   dB_z, dB_r, dB_h
  float* dP;     // [3][H][F]
  float* dcg;    // [3][H]
  float* dM0;    // [H][F]
  float* dM1;    // [R][H][F]
  float* dc0;    // [H]
  float* dprobs; // [T]
  float* hpart;  // fused-head per-CTA partials
  float* part;   // split-K partials
  size_t part_floats;
  int32_t* m1cp; // [R+1] chunk table of the per-region dM1 reduction (cell.cu k_m1_chunks)
  // tensor-core path (precision != FP32): weight images, tile-layout planes, per-CTA partials
  unsigned char* tc_img_f;   // forward weight image
  unsigned char* tc_img_b;   // backward weight image
  float *Zp, *Rp, *Hcp, *dhp_p;  // [T][nqt][H/4][128][4]
  float* Xt;                 // [T][BN][F] period-major copy of x (S and U are period-major too)
  float* hid_part;           // [T (max t-chunks)][nqt][H/4][128][4]
  float* tc_wpart;           // [TC_MAX_CTAS][TC_WPART_FLOATS]
  float* tc_dpp;             // [T * nqt] attention-gradient partials
  float* xw;                 // [B][x_rows][REGT_F][T]  x widened with zero features (fp32 / unfused tf32x3 paths when the
                             // caller's F < REGT_F; written by every forward, read by its backward), else NULL
  float* inv_c;              // [B] 1 / valid count per snapshot (loss_masked), written by k_loss_inv; NULL without y
  unsigned int* lc_part;     // [B][LC_CHUNKS] valid counts of each snapshot's chunks (k_loss_count); NULL without y
  size_t total;
};
constexpr int TC_MAX_CTAS = 160;
constexpr int LC_CHUNKS = 64;     // most blocks k_loss_count gives one snapshot
constexpr int TC_IMG_BYTES = 160 * 1024;
constexpr int F_IMG_BYTES = 432 * 1024;   // fused 3xTF32 cell (cell_f.cu): 12 ring stages of 32 KB + F-wide weights + constants at H = 128

Layout make_layout(const regt_args* a, void* base);

// features per node of the caller's x and [H, F] parameters (regt_args.F, 0 = REGT_F)
inline int feat_in(const regt_args* a) { return a->F > 0 ? a->F : REGT_F; }
// x as the FFMA and unfused tf32x3 kernels read it: REGT_F features per row
inline const float* x_wide(const regt_args* a, const Layout& L) { return L.xw ? L.xw : a->x; }

constexpr int HEAD_HID = 128;  // hidden_dim of the decoder MLP (models/RegionalTemporalGCN.py:19)
constexpr int WGRAD_SPLITS = 64;

// ---- host functions one file calls in another ----------------------------------------
// cell and head of each path (api.cu dispatches on Layout::route)
int cell_forward_fp32(const regt_args* a, const Layout& L, cudaStream_t st);    // cell.cu
int cell_backward_fp32(const regt_args* a, const Layout& L, cudaStream_t st);
int cell_forward_g(const regt_args* a, const Layout& L, cudaStream_t st);       // cell_g.cu
int cell_backward_g(const regt_args* a, const Layout& L, cudaStream_t st);
int cell_forward_f(const regt_args* a, const Layout& L, cudaStream_t st);       // cell_f.cu
int cell_backward_f(const regt_args* a, const Layout& L, cudaStream_t st);
int cell_forward_tc(const regt_args* a, const Layout& L, cudaStream_t st);      // cell_tc.cu
int cell_backward_tc(const regt_args* a, const Layout& L, cudaStream_t st);
size_t cell_backward_x_scratch_bytes(const regt_args* a, const regt_xgrad_plan* xp);   // input_grad.cu
int cell_backward_x(const regt_args* a, const Layout& L, const regt_xgrad_plan* xp, float* d_x, void* scratch, cudaStream_t st);
int head_forward(const regt_args* a, const Layout& L, cudaStream_t st);         // head.cu
int head_backward(const regt_args* a, const Layout& L, cudaStream_t st);
int head_forward_f(const regt_args* a, const Layout& L, cudaStream_t st);       // head_f.cu
int head_backward_f(const regt_args* a, const Layout& L, cudaStream_t st);
int head_forward_tc(const regt_args* a, const Layout& L, cudaStream_t st);      // head_tc.cu
LossX make_lossx(const regt_args* a, const Layout& L);                          // head.cu: the LossX of an LX head kernel

// weights.cu: collapsed weights before the cell, chain rule back to the parameters after it
int launch_prep(const regt_args* a, const Layout& L, cudaStream_t st);
int launch_chain(const regt_args* a, const Layout& L, cudaStream_t st);
// spmm.cu: F-wide SpMM on rows of `width` floats; period-major Xt / St / Ut of the tensor-core cells
int launch_spmm_rows(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y, int B,
                     int n_out, int n_in, int width, cudaStream_t st);
// x [B][xN][Fin][T]; Xt / St / Ut rows are REGT_F wide (features Fin.. are zeros)
// cell_f.cu: Feat [BNp][32] = 0 with column 16 = 1 in rows < BN (the ones column of the head's bias sums)
int launch_ones_f(int BN, int BNp, float* Feat, cudaStream_t st);
int launch_feat_tc(const regt_graph_plan& p, const float* x, int Fin, int B, int xN, int T, float* Xt, float* St, float* Ut,
                   cudaStream_t st);
// L.xw = x with zero features Fin..REGT_F-1 (no launch when L.xw is NULL)
int launch_widen_x(const regt_args* a, const Layout& L, cudaStream_t st);
// cell.cu
struct TNBatch;   // gemm_simt.cuh
int launch_wgrad_tn(const TNBatch& batch, long long rows, int splits, cudaStream_t st);   // split-K C = A^T B per problem of the batch
// out[i] (+)= sum_s part[s*count + i]
int launch_reduce_splits(const float* part, float* out, long long count, int splits, int accumulate, cudaStream_t st);
// part[s][c] = sum over the rows of split s of A[r*lda + c]
int launch_colsum(const float* A, int lda, int C, long long rows, int splits, float* part, cudaStream_t st);
int launch_wgrad_m1(const regt_args* a, const Layout& L, cudaStream_t st);      // dM1 per region from the row-major gate gradients
int launch_wgrad_m1_kt(const regt_args* a, const Layout& L, cudaStream_t st);   // ... from the transposed tiles of the fused backward
// cell_g.cu: d probs from the fused backward's fp64 partials; F-wide weight gradients from the [splits][4H][32] partials of D^T Feat
int launch_f_sum_dpp(const double* part, int nparts, int T, float* dprobs, cudaStream_t st);
int launch_fw_scatter(const float* Cp, int splits, int H, const Layout& L, cudaStream_t st);
// gemm_tma.cu: TMA-fed 3xTF32 GEMMs and their single-pass bf16 forms
enum class GemmKind { Tf32x3, Bf16 };
size_t gemm_nt_scratch_floats(int N, int K, GemmKind kind);   // hi | lo images of the weight operand, or its bf16 image
int launch_gemm_nt_tma(const float* A, long long lda, const float* Bt, long long ldb, float* C, long long ldc, long long M, int N,
                       int K, float* scratch, cudaStream_t st, GemmKind kind = GemmKind::Tf32x3);
int launch_gemm_tn(const float* A, long long lda, const float* B, long long ldb, float* Cp, long long M, int K, int N, int splits,
                   cudaStream_t st, const float* B2, long long ldb2, float* Cp2, long long c2_split, int relu_b,
                   GemmKind kind = GemmKind::Tf32x3);
int launch_gemm_tn_tma(const float* A, long long lda, long long M, int Ktot, int nseg, const int* seg_k0, const int* seg_b,
                       float* const* seg_C, const float* const* Bs, const long long* ldbs, int N, int splits, const float* B2,
                       long long ldb2, float* C2, long long c2_split, cudaStream_t st, int relu_b, GemmKind kind = GemmKind::Tf32x3);
int launch_gemm_kt(const float* AT, long long ntile, int Ktot, int nseg, const int* seg_k0, const int* seg_k1, const int* seg_b,
                   float* const* seg_C, const float* const* BTs, int N, int splits, const float* FT, float* C2, long long c2_split,
                   cudaStream_t st);
// head.cu / head_tc.cu: the fused heads' per-CTA partials and their cross-CTA sum
int head_part_stride_host(int H, int O);
int launch_head_grad_reduce(const regt_args* a, const Layout& L, cudaStream_t st);
int launch_head_dw1_tf32x3(const regt_args* a, const Layout& L, const float* ones, cudaStream_t st);
int head_tc_grid(const regt_args* a);
// cell_tc.cu: period chunks of the bf16 forward (the partials of out_hidden it leaves)
int tc_num_chunks(const regt_args* a);

}  // namespace regt
