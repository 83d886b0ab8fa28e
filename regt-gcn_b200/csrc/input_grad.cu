// Gradient wrt x of the cell (regt_cell_backward_x, include/regt_b200.h), on the fp32 and tf32x3 paths.
//
// The cell sees x only through three F-wide linear maps (cell.cu header): S = A_hat X feeds the three gates through the
// first F rows of Wzr / Wc, X itself and U_seg = L_hat_r X feed the regional combine through M0 / M1[r].  So
//   dx = dXd + A_hat^T dS + sum_r C_r^T dU,
// with the F-wide row gradients contracted from the gate-gradient plane D = [Dz | Dr | Dc | Dpre] the cell backward left in
// the workspace.  Three passes:
//   1. k_xg_contract: one pass over D (4H floats per row and period), 40 H FFMA per row against [4H][F] weights in shared
//      memory.  Writes G [B][2N + nseg][T][F]: stacked rows dXd | dS | dU of a snapshot, the F values of a (row, period)
//      contiguous -- one 32-byte sector per thread and period.
//   2. the transposed operator (regt_xgrad_plan) on the F*T-wide rows of G with the F-wide SpMM of the forward
//      (launch_spmm_rows, n_in = 2N + nseg > n_out = N): sequential CSR order, no atomics -> bit-reproducible.
//   3. k_xg_layout: [B][N][T][F] -> x's layout [B][N][Fin][T] (the caller's Fin <= F features; the padded ones are dropped).
// Keeping the period inside the SpMM row (width F*T, as in the forward) keeps the SpMM kernels' lanes busy; rows of F = 8
// floats would use 2 of a warp's 32 lanes.
#include "common.cuh"

namespace regt {

constexpr int F = REGT_F;

struct XgK {
  const float* D;          // gate-gradient plane (layout: TILED below)
  const float *Wzr, *Wc;   // collapsed gate weights; rows 0..F-1 are (A_g W_g)^T
  const float* M0t;        // [F][H]
  const float* M1h;        // [R][H][F]  (M1t transposed: the F weights of a column are one 32-byte row)
  const int32_t *seg_ptr, *seg_reg;
  float* G;                // [B][n_src][T][F]
  long long BN, rows;      // B*N, B*N*T
  int N, T, H, nqt, n_src, mode;
};

// M1h[r][j][f] = M1t[r][f][j]
__global__ void k_xg_m1h(const float* __restrict__ M1t, int R, int H, float* __restrict__ M1h) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)R * H * F) return;
  const int f = (int)(i % F);
  const long long rj = i / F;
  const int j = (int)(rj % H), r = (int)(rj / H);
  M1h[i] = M1t[((size_t)r * F + f) * H + j];
}

__device__ __forceinline__ void st8(float* p, const float (&v)[F]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}

// One thread per (row, period).  TILED: D is the fused backward's transposed tiles [T*nqt][4 row quarters][4H][32 rows]; a
// block is one (period, 128-row tile), warp = row quarter, lane = row, so every column read is one 128-byte line.  Rows
// at or past B*N (pad rows of the last tile) are never read.  Row-major: D is [rows][4H], row = q*T + t, a block is 128
// consecutive rows and a thread reads its row in float4 pieces.  Weights: Ws[c][f] (c < 3H: the dS weights, c >= 3H: M0)
// in shared memory, read as warp-wide broadcasts; M1h rows through L1 (a warp's rows are neighbouring nodes, nearly always
// in one region).
template <bool TILED>
__global__ void __launch_bounds__(128) k_xg_contract(XgK k) {
  extern __shared__ __align__(16) float Ws[];   // [4H][F]
  const int H = k.H, tid = threadIdx.x;
  for (int i = tid; i < 4 * H * F; i += 128) {
    const int c = i / F, f = i - c * F;
    Ws[i] = c < 2 * H ? k.Wzr[(size_t)f * 2 * H + c] : (c < 3 * H ? k.Wc[(size_t)f * H + c - 2 * H] : k.M0t[(size_t)f * H + c - 3 * H]);
  }
  __syncthreads();
  long long q;
  int t;
  const float* dp;
  if (TILED) {
    const int tp = blockIdx.x, qt = tp % k.nqt;
    t = tp / k.nqt;
    q = (long long)qt * 128 + tid;
    dp = k.D + ((size_t)tp * 4 + (tid >> 5)) * (size_t)(4 * H * 32) + (tid & 31);
    if (q >= k.BN) return;
  } else {
    const long long row = (long long)blockIdx.x * 128 + tid;
    if (row >= k.rows) return;
    q = row / k.T;
    t = (int)(row - q * k.T);
    dp = k.D + (size_t)row * 4 * H;
  }
  auto load8 = [&](int c0, float (&d)[8]) {
    if (TILED) {
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] = __ldg(dp + (size_t)(c0 + i) * 32);
    } else {
      const float4 a = __ldg(reinterpret_cast<const float4*>(dp + c0)), b = __ldg(reinterpret_cast<const float4*>(dp + c0 + 4));
      d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.w; d[4] = b.x; d[5] = b.y; d[6] = b.z; d[7] = b.w;
    }
  };
  auto fma8 = [](float dv, float4 w0, float4 w1, float (&acc)[F]) {
    acc[0] = fmaf(dv, w0.x, acc[0]); acc[1] = fmaf(dv, w0.y, acc[1]); acc[2] = fmaf(dv, w0.z, acc[2]); acc[3] = fmaf(dv, w0.w, acc[3]);
    acc[4] = fmaf(dv, w1.x, acc[4]); acc[5] = fmaf(dv, w1.y, acc[5]); acc[6] = fmaf(dv, w1.z, acc[6]); acc[7] = fmaf(dv, w1.w, acc[7]);
  };
  const float4* W4 = reinterpret_cast<const float4*>(Ws);
  // dS = Dz . (A_z W_z) + Dr . (A_r W_r) + Dc . (A_c W_c)
  float s[F] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
  for (int c0 = 0; c0 < 3 * H; c0 += 8) {
    float d[8];
    load8(c0, d);
#pragma unroll
    for (int i = 0; i < 8; ++i) fma8(d[i], W4[(c0 + i) * 2], W4[(c0 + i) * 2 + 1], s);
  }
  const int b = (int)(q / k.N), n = (int)(q - (long long)b * k.N);
  const size_t gb = (size_t)b * k.n_src;
  auto out = [&](int srow) { return k.G + ((gb + srow) * k.T + t) * F; };
  st8(out(k.N + n), s);
  // dXd = Dpre . M0 and dU = Dpre . M1[r] for the node's first segment in the same pass; further segments (a node in
  // several regional lists) take one more pass over Dpre each.  The bare TGCN cell has no Chebyshev branch: zeros.
  const bool cheb = k.mode != REGT_MODE_TGCN;
  const int sb = k.seg_ptr ? k.seg_ptr[n] : 0, se = k.seg_ptr ? k.seg_ptr[n + 1] : 0;
  float xd[F] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float u[F] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (cheb) {
    const float4* m1 = reinterpret_cast<const float4*>(k.M1h + (size_t)(se > sb ? k.seg_reg[sb] : 0) * H * F);
#pragma unroll 1
    for (int j0 = 0; j0 < H; j0 += 8) {
      float d[8];
      load8(3 * H + j0, d);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        fma8(d[i], W4[(3 * H + j0 + i) * 2], W4[(3 * H + j0 + i) * 2 + 1], xd);
        fma8(d[i], __ldg(m1 + (j0 + i) * 2), __ldg(m1 + (j0 + i) * 2 + 1), u);
      }
    }
  }
  st8(out(n), xd);
  for (int sg = sb; sg < se; ++sg) {
    if (cheb && sg > sb) {
      const float4* m1 = reinterpret_cast<const float4*>(k.M1h + (size_t)k.seg_reg[sg] * H * F);
#pragma unroll
      for (int f = 0; f < F; ++f) u[f] = 0.f;
#pragma unroll 1
      for (int j0 = 0; j0 < H; j0 += 8) {
        float d[8];
        load8(3 * H + j0, d);
#pragma unroll
        for (int i = 0; i < 8; ++i) fma8(d[i], __ldg(m1 + (j0 + i) * 2), __ldg(m1 + (j0 + i) * 2 + 1), u);
      }
    }
    st8(out(2 * k.N + sg), u);
  }
}

// dx[q][f][t] = Y[q][t][f] for the caller's Fin features (dx [B*N][Fin][T]; the padded ones are dropped)
__global__ void k_xg_layout(const float* __restrict__ Y, int Fin, int T, long long total, float* __restrict__ dx) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long q = i / ((long long)Fin * T);
  const int rem = (int)(i - q * Fin * T), f = rem / T, t = rem - f * T;
  dx[i] = __ldg(Y + (q * T + t) * F + f);
}

struct XgScratch {
  float *G, *Y, *M1h;
  size_t total;
};
static XgScratch xg_scratch(const regt_args* a, const regt_xgrad_plan* xp, void* base) {
  XgScratch s{};
  Carver c(base);
  const size_t B = a->B, T = a->T, R = a->plan.R > 0 ? a->plan.R : 1;
  s.G = c.take<float>(B * (size_t)xp->n_src * T * F);
  s.Y = c.take<float>(B * (size_t)a->N * T * F);
  s.M1h = c.take<float>(R * a->H * F);
  s.total = align_up(c.off, 256);
  return s;
}
size_t cell_backward_x_scratch_bytes(const regt_args* a, const regt_xgrad_plan* xp) { return xg_scratch(a, xp, nullptr).total; }

int cell_backward_x(const regt_args* a, const Layout& L, const regt_xgrad_plan* xp, float* d_x, void* scratch, cudaStream_t st) {
  const int H = a->H, T = a->T, R = a->plan.R > 0 ? a->plan.R : 1;
  const XgScratch S = xg_scratch(a, xp, scratch);
  const bool tiled = L.route.cell == CellPath::Tf32x3Fused;   // D as the fused backward's transposed tiles
  XgK k{};
  k.D = L.D; k.Wzr = L.Wzr; k.Wc = L.Wc; k.M0t = L.M0t; k.M1h = S.M1h;
  k.seg_ptr = a->plan.nseg > 0 ? a->plan.seg_ptr : nullptr;
  k.seg_reg = a->plan.seg_reg;
  k.G = S.G;
  k.BN = (long long)a->B * a->N;
  k.rows = k.BN * T;
  k.N = a->N; k.T = T; k.H = H; k.nqt = (int)((k.BN + 127) / 128); k.n_src = xp->n_src; k.mode = a->mode;
  if (a->mode != REGT_MODE_TGCN) {
    k_xg_m1h<<<cdiv((long long)R * H * F, 256), 256, 0, st>>>(L.M1t, R, H, S.M1h);
    REGT_LAUNCHED("k_xg_m1h", st);
  }
  const size_t smem = (size_t)4 * H * F * sizeof(float);
  if (tiled) {
    REGT_CUDA(cudaFuncSetAttribute(k_xg_contract<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_xg_contract<true><<<(unsigned)(k.nqt * (long long)T), 128, smem, st>>>(k);
  } else {
    REGT_CUDA(cudaFuncSetAttribute(k_xg_contract<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_xg_contract<false><<<cdiv(k.rows, 128), 128, smem, st>>>(k);
  }
  REGT_LAUNCHED("k_xg_contract", st);
  if (launch_spmm_rows(xp->rowptr, xp->col, xp->val, S.G, S.Y, a->B, a->N, xp->n_src, F * T, st)) return -1;
  const long long total = k.BN * feat_in(a) * T;
  k_xg_layout<<<cdiv(total, 256), 256, 0, st>>>(S.Y, feat_in(a), T, total, d_x);
  REGT_LAUNCHED("k_xg_layout", st);
  return 0;
}

}  // namespace regt
