// REGT_PREC_TF32X3 and REGT_PREC_BF16 for any hidden width that is a multiple of 32: the regional temporal GCN
// cell with every H x H contraction on the sm_100a tensor cores through the generic GEMMs of gemm_tma.cu, forward AND
// backward -- 3xTF32 (fp32-equivalent accuracy) or single-pass bf16 (Route::cell Bf16Gemm, the bf16 tolerance), the
// only part of this file that depends on the precision.  The elementwise passes and saved planes are fp32 in both.  Unlike the fused H = 64 kernels of cell_tc.cu the
// gate pre-activations make one round trip through HBM, which is what lets the same code serve H = 128
// (configs 4, 5) and H = 256 (configs 1, 3): no weight set has to fit one SM's shared memory or TMEM.
//
// Planes are the fp32 path's (row = (b*N+n)*T + t; cell.cu), so the F-wide weight gradients, the
// attention kernels and the chain rule are shared with it.  Reference arithmetic replaced:
// models/utils.py:163-203, models/RegionalTemporalGCN.py:134-148, models/TemporalGCN.py:84-90.
//
//   forward   h   = act(X M0 + U M1 + c0)                          k_g_h        (F-wide, CUDA cores)
//             Pzr = h . [B_z | B_r]^T                              gemm_nt x2   (tensor cores; B_g = linear_g.weight[:, H:])
//             Z,R = sigmoid(Pzr + S Pzr_s + czr), hR = h*R          k_g_zr
//             Pc  = hR . B_h^T                                      gemm_nt
//             H~  = tanh(Pc + S Pc_s + cc), H' = Z h + (1-Z) H~,    k_g_c  (period-attention sum in registers)
//             out_hidden = sum_t probs[t] H'
//   backward  Dz, Dh from G, probs, saved planes; d probs         k_g_b1
//             dHR = Dh . B_h                                        gemm_nt (B_h^T packed by k_g_pack_bt)
//             Dr  = dHR h R (1-R)                                   k_g_b2
//             dhg = [Dz | Dr] . [B_z ; B_r]                         gemm_nt
//             dhp = act'(h) (probs G Z + dHR R + dhg)               k_g_b3
//             dB_z, dB_r = [Dz|Dr]^T h ;  dB_h = Dh^T hR            gemm_tn (row contraction, split over rows)
//             dP_g, dc_g, dM0, dc0 = D^T [S | X | 1]                gemm_tn on the 32-wide feature plane (k_g_feat)
#include "common.cuh"
#include "gemm_simt.cuh"

namespace regt {

constexpr int F = REGT_F;

namespace {
struct GK {
  long long rows;
  int N, xN, T, H, nseg, mode;
  const float *x, *S, *U, *h_ext;
  const int32_t *seg_ptr, *seg_reg;
  const float *M0t, *M1t, *c0, *Wzr, *Wc, *czr, *cc, *probs, *G;
  float *h, *Z, *Rg, *Hc, *hR, *Hn, *D;
  float* d_h_ext;
  float* Feat;        // [rows][32]: S_t (8) | X_t (8) | 1 | 0...   B operand of the F-wide weight-gradient GEMM
  float* out_hidden;  // [BN][H]
  double* dp_part;    // [gridDim.x][T] attention-gradient partials (fp64: the softmax Jacobian differences them)
  long long BN;
};

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
// one thread = (row, 4 consecutive columns)
__device__ __forceinline__ bool rowcol(const GK& a, long long& row, int& j) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int H4 = a.H >> 2;
  row = i / H4;
  j = (int)(i - row * H4) * 4;
  return row < a.rows;
}
__device__ __forceinline__ float sigm(float v) { return 1.0f / (1.0f + expf(-v)); }

// one thread = (q = b*N+n, 4 consecutive columns), walking the T periods of the row block: the F-wide weight
// columns it needs are loaded ONCE into registers, the x / S / U values of a period are warp-uniform broadcasts
__device__ __forceinline__ bool qcol(const GK& a, long long i, long long& q, int& j) {
  const int H4 = a.H >> 2;
  q = i / H4;
  j = (int)(i - q * H4) * 4;
  return q < a.BN;
}
__device__ __forceinline__ void fma4(float s, const float4& w, float (&v)[4]) {
  v[0] = fmaf(s, w.x, v[0]); v[1] = fmaf(s, w.y, v[1]); v[2] = fmaf(s, w.z, v[2]); v[3] = fmaf(s, w.w, v[3]);
}

// h = act(X_t M0 + sum_seg U_seg,t M1[region] + c0)      (regional combine on the F-wide features)
__global__ void __launch_bounds__(256) k_g_h(GK a) {
  long long q; int j;
  if (!qcol(a, blockIdx.x * (long long)blockDim.x + threadIdx.x, q, j)) return;
  const int H = a.H, T = a.T;
  if (a.mode == REGT_MODE_TGCN) {
    for (int t = 0; t < T; ++t) {
      const long long row = q * T + t;
      const float4 e = a.h_ext ? ld4(a.h_ext + row * H + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      st4(a.h + row * H + j, e.x, e.y, e.z, e.w);
    }
    return;
  }
  const int b = (int)(q / a.N), n = (int)(q - (long long)b * a.N);
  const float* xr = a.x + ((size_t)b * a.xN + n) * F * T;
  const float4 c = ld4(a.c0 + j);
  float4 w0[F], w1[F];
#pragma unroll
  for (int f = 0; f < F; ++f) w0[f] = ld4(a.M0t + f * H + j);
  const int s0 = a.seg_ptr[n], s1 = a.seg_ptr[n + 1];
  const float* u0 = nullptr;
  if (s1 > s0) {   // the node's first (normally only) regional segment: its M1 block stays in registers too
    u0 = a.U + ((size_t)b * a.nseg + s0) * F * T;
    const float* m = a.M1t + (size_t)a.seg_reg[s0] * F * H + j;
#pragma unroll
    for (int f = 0; f < F; ++f) w1[f] = ld4(m + f * H);
  }
  for (int t = 0; t < T; ++t) {
    float v[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
    for (int f = 0; f < F; ++f) fma4(__ldg(xr + f * T + t), w0[f], v);
    if (u0) {
#pragma unroll
      for (int f = 0; f < F; ++f) fma4(__ldg(u0 + f * T + t), w1[f], v);
    }
    for (int s = s0 + 1; s < s1; ++s) {   // a node that appears in several regional lists (random decomposition)
      const float* ur = a.U + ((size_t)b * a.nseg + s) * F * T + t;
      const float* m = a.M1t + (size_t)a.seg_reg[s] * F * H + j;
#pragma unroll
      for (int f = 0; f < F; ++f) fma4(__ldg(ur + f * T), ld4(m + f * H), v);
    }
    if (a.mode == REGT_MODE_REGIONAL) {
#pragma unroll
      for (int e = 0; e < 4; ++e) v[e] = v[e] > 0.f ? v[e] : 0.01f * v[e];   // F.leaky_relu
    }
    st4(a.h + (q * T + t) * H + j, v[0], v[1], v[2], v[3]);
  }
}

// the F-wide part of a gate pre-activation: sum_f S[q][f][t] * W[f][n0 + e] for 4 columns
__device__ __forceinline__ void s_part(const float* __restrict__ S, long long q, int t, int T, const float* __restrict__ W, int ldw,
                                       int n, float (&v)[4]) {
  const float* sr = S + q * F * T + t;
#pragma unroll
  for (int f = 0; f < F; ++f) {
    const float sv = __ldg(sr + f * T);
    const float4 w = ld4(W + (size_t)f * ldw + n);
    v[0] = fmaf(sv, w.x, v[0]); v[1] = fmaf(sv, w.y, v[1]); v[2] = fmaf(sv, w.z, v[2]); v[3] = fmaf(sv, w.w, v[3]);
  }
}

// Z, R = sigmoid(Pzr + S Wzr_s + czr) ; hR = h * R         Pzr = D[:, 0:2H]
__global__ void __launch_bounds__(256) k_g_zr(GK a) {
  long long row; int j;
  if (!rowcol(a, row, j)) return;
  const int H = a.H, T = a.T;
  const long long q = row / T;
  const int t = (int)(row - q * T);
  const float4 pz = ld4(a.D + row * 4 * H + j), pr = ld4(a.D + row * 4 * H + H + j);
  const float4 bz = ld4(a.czr + j), br = ld4(a.czr + H + j);
  float z[4] = {pz.x + bz.x, pz.y + bz.y, pz.z + bz.z, pz.w + bz.w};
  float r[4] = {pr.x + br.x, pr.y + br.y, pr.z + br.z, pr.w + br.w};
  s_part(a.S, q, t, T, a.Wzr, 2 * H, j, z);
  s_part(a.S, q, t, T, a.Wzr, 2 * H, H + j, r);
  const float4 hv = ld4(a.h + row * H + j);
#pragma unroll
  for (int e = 0; e < 4; ++e) { z[e] = sigm(z[e]); r[e] = sigm(r[e]); }
  st4(a.Z + row * H + j, z[0], z[1], z[2], z[3]);
  st4(a.Rg + row * H + j, r[0], r[1], r[2], r[3]);
  st4(a.hR + row * H + j, hv.x * r[0], hv.y * r[1], hv.z * r[2], hv.w * r[3]);
}

// H~ = tanh(Pc + S Wc_s + cc) ; H' = Z h + (1 - Z) H~ ; out_hidden = sum_t probs[t] H'      Pc = D[:, 2H:3H]
// (the period-attention sum of models/RegionalTemporalGCN.py:134,146 stays in registers: no H' plane)
__global__ void __launch_bounds__(256) k_g_c(GK a) {
  long long q; int j;
  if (!qcol(a, blockIdx.x * (long long)blockDim.x + threadIdx.x, q, j)) return;
  const int H = a.H, T = a.T;
  const float4 bc = ld4(a.cc + j);
  float4 wc[F];
#pragma unroll
  for (int f = 0; f < F; ++f) wc[f] = ld4(a.Wc + (size_t)f * H + j);
  const float* sr = a.S + q * F * T;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t = 0; t < T; ++t) {
    const long long row = q * T + t;
    const float4 pc = ld4(a.D + row * 4 * H + 2 * H + j);
    float c[4] = {pc.x + bc.x, pc.y + bc.y, pc.z + bc.z, pc.w + bc.w};
#pragma unroll
    for (int f = 0; f < F; ++f) fma4(__ldg(sr + f * T + t), wc[f], c);
    const float4 hv = ld4(a.h + row * H + j), zv = ld4(a.Z + row * H + j);
    const float h[4] = {hv.x, hv.y, hv.z, hv.w}, z[4] = {zv.x, zv.y, zv.z, zv.w};
    const float p = __ldg(a.probs + t);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      c[e] = tanhf(c[e]);
      acc[e] = fmaf(p, z[e] * h[e] + (1.0f - z[e]) * c[e], acc[e]);
    }
    st4(a.Hc + row * H + j, c[0], c[1], c[2], c[3]);
  }
  st4(a.out_hidden + q * H + j, acc[0], acc[1], acc[2], acc[3]);
}

// Feat[row] = S_t | X_t | 1 | 0   (32 floats per row)
__global__ void __launch_bounds__(256) k_g_feat(GK a) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long row = i >> 3;
  if (row >= a.rows) return;
  const int c4 = (int)(i & 7), T = a.T;
  const long long q = row / T;
  const int t = (int)(row - q * T);
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (c4 < 2) {
    const float* sr = a.S + q * F * T + (4 * c4) * T + t;
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = __ldg(sr + e * T);
  } else if (c4 < 4) {
    const int b = (int)(q / a.N), n = (int)(q - (long long)b * a.N);
    const float* xr = a.x + ((size_t)b * a.xN + n) * F * T + (4 * (c4 - 2)) * T + t;
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = __ldg(xr + e * T);
  } else if (c4 == 4) {
    v[0] = 1.0f;
  }
  st4(a.Feat + row * 32 + 4 * c4, v[0], v[1], v[2], v[3]);
}

// Dz -> D[:, 0:H], Dh -> D[:, 2H:3H]; attention gradient partials d probs[t] = sum G * H'_t (H' recomputed)
__global__ void __launch_bounds__(256) k_g_b1(GK a) {
  __shared__ double red[8][64];
  const int H = a.H, T = a.T, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long total = a.BN * (H >> 2);
  for (int t = threadIdx.x; t < 8 * 64; t += 256) (&red[0][0])[t] = 0.0;
  __syncthreads();
  // grid-stride over (q, 4 columns); trip counts are warp-uniform up to the tail (idle lanes add zeros)
  for (long long base = blockIdx.x * (long long)blockDim.x; base < total; base += (long long)gridDim.x * blockDim.x) {
    long long q; int j;
    const bool live = qcol(a, base + threadIdx.x, q, j);
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) g = ld4(a.G + q * H + j);
    const float gr[4] = {g.x, g.y, g.z, g.w};
    for (int t = 0; t < T; ++t) {
      float dp = 0.f;
      if (live) {
        const long long row = q * T + t;
        const float p = __ldg(a.probs + t);
        const float4 hv = ld4(a.h + row * H + j), zv = ld4(a.Z + row * H + j), cv = ld4(a.Hc + row * H + j);
        const float h[4] = {hv.x, hv.y, hv.z, hv.w}, z[4] = {zv.x, zv.y, zv.z, zv.w}, c[4] = {cv.x, cv.y, cv.z, cv.w};
        float dz[4], dh[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float gg = p * gr[e];                       // dH' = probs[t] * d out_hidden
          dp = fmaf(gr[e], z[e] * h[e] + (1.0f - z[e]) * c[e], dp);
          dz[e] = gg * (h[e] - c[e]) * z[e] * (1.0f - z[e]);
          dh[e] = gg * (1.0f - z[e]) * (1.0f - c[e] * c[e]);
        }
        st4(a.D + row * 4 * H + j, dz[0], dz[1], dz[2], dz[3]);
        st4(a.D + row * 4 * H + 2 * H + j, dh[0], dh[1], dh[2], dh[3]);
      }
      double dpd = (double)dp;               // four terms in fp32, everything above in fp64
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) dpd += __shfl_xor_sync(0xffffffffu, dpd, d);
      if (lane == 0) red[warp][t] += dpd;    // only this warp's lane 0 touches red[warp][*]: fixed order
    }
  }
  __syncthreads();
  if (threadIdx.x < T) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    a.dp_part[(size_t)blockIdx.x * T + threadIdx.x] = s;
  }
}

// Dr = dHR * h * R (1 - R) -> D[:, H:2H]                   dHR = Hn plane (reused)
__global__ void __launch_bounds__(256) k_g_b2(GK a) {
  long long row; int j;
  if (!rowcol(a, row, j)) return;
  const int H = a.H;
  const float4 d = ld4(a.Hn + row * H + j), hv = ld4(a.h + row * H + j), rv = ld4(a.Rg + row * H + j);
  st4(a.D + row * 4 * H + H + j, d.x * hv.x * rv.x * (1.0f - rv.x), d.y * hv.y * rv.y * (1.0f - rv.y),
      d.z * hv.z * rv.z * (1.0f - rv.z), d.w * hv.w * rv.w * (1.0f - rv.w));
}

// d h = probs G Z + dHR R + dhg ; through the regional combine's activation -> D[:, 3H:4H] (in place over dhg)
__global__ void __launch_bounds__(256) k_g_b3(GK a) {
  long long row; int j;
  if (!rowcol(a, row, j)) return;
  const int H = a.H, T = a.T;
  const long long q = row / T;
  const int t = (int)(row - q * T);
  const float p = __ldg(a.probs + t);
  const float4 g = ld4(a.G + q * H + j), zv = ld4(a.Z + row * H + j), d = ld4(a.Hn + row * H + j), rv = ld4(a.Rg + row * H + j);
  const float4 dg = ld4(a.D + row * 4 * H + 3 * H + j);
  float v[4] = {fmaf(d.x, rv.x, p * g.x * zv.x) + dg.x, fmaf(d.y, rv.y, p * g.y * zv.y) + dg.y,
                fmaf(d.z, rv.z, p * g.z * zv.z) + dg.z, fmaf(d.w, rv.w, p * g.w * zv.w) + dg.w};
  if (a.mode == REGT_MODE_TGCN) {
    if (a.d_h_ext) st4(a.d_h_ext + row * H + j, v[0], v[1], v[2], v[3]);
    v[0] = v[1] = v[2] = v[3] = 0.f;
  } else if (a.mode == REGT_MODE_REGIONAL) {
    const float4 hv = ld4(a.h + row * H + j);
    v[0] *= hv.x > 0.f ? 1.0f : 0.01f; v[1] *= hv.y > 0.f ? 1.0f : 0.01f;
    v[2] *= hv.z > 0.f ? 1.0f : 0.01f; v[3] *= hv.w > 0.f ? 1.0f : 0.01f;
  }
  st4(a.D + row * 4 * H + 3 * H + j, v[0], v[1], v[2], v[3]);
}

// K-major B operands of the data-gradient GEMMs: BhT[k][n] = B_h[n][k], BzrT[k][g*H + n] = B_g[n][k]
__global__ void k_g_pack_bt(const float* __restrict__ lw0, const float* __restrict__ lw1, const float* __restrict__ lw2, int H,
                            float* __restrict__ BhT, float* __restrict__ BzrT) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 3 * H * H) return;
  const int g = i / (H * H), rem = i % (H * H), k = rem / H, n = rem % H;   // n fastest: coalesced writes
  const float* lw = g == 0 ? lw0 : (g == 1 ? lw1 : lw2);
  const float v = __ldg(lw + (size_t)n * 2 * H + H + k);
  if (g == 2) BhT[(size_t)k * H + n] = v;
  else BzrT[(size_t)k * 2 * H + g * H + n] = v;
}

// out[i] = sum over nparts of part[p * stride + i]   (fixed order; 32 outputs x 8 partial subsets per block)
__global__ void __launch_bounds__(256) k_g_sum_parts(const float* __restrict__ part, int stride, int nparts, int n, float* __restrict__ out) {
  __shared__ float red[8][32];
  const int i = blockIdx.x * 32 + threadIdx.x;
  const float s = sum_parts_32x8(part, (size_t)stride, nparts, i, i < n, red);
  if (threadIdx.y == 0 && i < n) out[i] = s;
}
// Cp[split][4H][32] = D^T . Feat  ->  dP_g = D_g^T S, dc_g, dM0 = dhp^T X, dc0      (what k_skinny_reduce writes)
__global__ void __launch_bounds__(256) k_g_fw_scatter(const float* __restrict__ Cp, int splits, int H, float* __restrict__ dP,
                                                      float* __restrict__ dcg, float* __restrict__ dM0, float* __restrict__ dc0) {
  __shared__ float red[8][32];
  const int i = blockIdx.x * 32 + threadIdx.x;       // (c, col) with col = i & 31
  const int n = 4 * H * 32;
  const float s = sum_parts_32x8(Cp, (size_t)n, splits, i, i < n, red);
  if (threadIdx.y != 0 || i >= n) return;
  const int c = i >> 5, col = i & 31;
  if (c < 3 * H) {
    if (col < F) dP[(size_t)c * F + col] = s;
    else if (col == 16) dcg[c] = s;
  } else {
    const int m = c - 3 * H;
    if (col >= 8 && col < 16) dM0[(size_t)m * F + col - 8] = s;
    else if (col == 16) dc0[m] = s;
  }
}

// d probs[t] = sum over the CTAs of the fused backward's fp64 partials, in CTA order
__global__ void k_f_sum_dpp(const double* __restrict__ part, int nparts, int T, float* __restrict__ out) {
  const int t = threadIdx.x;
  if (t >= T) return;
  double s = 0.0;
  for (int p = 0; p < nparts; ++p) s += part[(size_t)p * T + t];
  out[t] = (float)s;
}

GK make_gk(const regt_args* a, const Layout& L) {
  GK k{};
  k.rows = (long long)a->B * a->N * a->T;
  k.N = a->N; k.xN = a->x_rows > 0 ? a->x_rows : a->N; k.T = a->T; k.H = a->H; k.nseg = a->plan.nseg; k.mode = a->mode;
  k.x = x_wide(a, L); k.S = L.S; k.U = L.U; k.h_ext = a->h_ext;
  k.seg_ptr = a->plan.seg_ptr; k.seg_reg = a->plan.seg_reg;
  k.M0t = L.M0t; k.M1t = L.M1t; k.c0 = L.c0; k.Wzr = L.Wzr; k.Wc = L.Wc; k.czr = L.czr; k.cc = L.cc; k.probs = L.probs;
  k.G = L.G;
  k.h = L.h; k.Z = L.Z; k.Rg = L.Rg; k.Hc = L.Hc; k.hR = L.hR; k.Hn = L.Hn; k.D = L.D;
  k.d_h_ext = a->d_h_ext;
  k.Feat = L.Feat; k.out_hidden = a->out_hidden; k.BN = (long long)a->B * a->N;
  return k;
}
#define G_LAUNCH(kern, name)                                                      \
  do {                                                                            \
    kern<<<cdiv(k.rows * (H / 4), 256), 256, 0, st>>>(k);                         \
    REGT_LAUNCHED(name, st);                                                      \
  } while (0)
}  // namespace

// shared with the fused backward of cell_f.cu
int launch_f_sum_dpp(const double* part, int nparts, int T, float* dprobs, cudaStream_t st) {
  k_f_sum_dpp<<<1, 64, 0, st>>>(part, nparts, T, dprobs);
  REGT_LAUNCHED("k_f_sum_dpp", st);
  return 0;
}
int launch_fw_scatter(const float* Cp, int splits, int H, const Layout& L, cudaStream_t st) {
  k_g_fw_scatter<<<cdiv(4ll * H * 32, 32), dim3(32, 8), 0, st>>>(Cp, splits, H, L.dP, L.dcg, L.dM0, L.dc0);
  REGT_LAUNCHED("k_g_fw_scatter", st);
  return 0;
}

// the GEMMs of this call: 3xTF32 or single-pass bf16
static GemmKind gemm_kind(const Layout& L) { return L.route.cell == CellPath::Bf16Gemm ? GemmKind::Bf16 : GemmKind::Tf32x3; }

int cell_forward_g(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, T = a->T;
  const long long BN = (long long)a->B * a->N;
  const int xN = a->x_rows > 0 ? a->x_rows : a->N;
  const GemmKind gk = gemm_kind(L);
  REGT_CHECK(T <= 64, "precision %s supports up to 64 periods (got %d)", gk == GemmKind::Bf16 ? "bf16" : "tf32x3", T);
  if (launch_prep(a, L, st)) return -1;
  if (launch_widen_x(a, L, st)) return -1;
  if (launch_spmm_rows(a->plan.g_rowptr, a->plan.g_col, a->plan.g_val, x_wide(a, L), L.S, a->B, a->N, xN, F * T, st)) return -1;
  if (a->mode != REGT_MODE_TGCN && a->plan.nseg > 0) {
    if (launch_spmm_rows(a->plan.seg_eptr, a->plan.c_col, a->plan.c_val, x_wide(a, L), L.U, a->B, a->plan.nseg, xN, F * T, st))
      return -1;
  }
  GK k = make_gk(a, L);
  k_g_h<<<cdiv(BN * (H / 4), 256), 256, 0, st>>>(k);
  REGT_LAUNCHED("k_g_h", st);
  // feature plane [S | X | 1]: F-wide input of the fused gate epilogues below, and second operand of the
  // weight-gradient contractions (cell and head backward)
  k_g_feat<<<cdiv(k.rows * 8, 256), 256, 0, st>>>(k);
  REGT_LAUNCHED("k_g_feat", st);
  // Pzr = h . [B_z | B_r]^T : the K-major B operand is the reference parameter itself (linear_g.weight[:, H:]).
  // (A gate epilogue inside this GEMM -- F-wide term as FMAs on the accumulator + sigmoid + h * R in the four epilogue
  // warps -- was built and measured in round 1: slower, 200 -> 231 ms at config 4.  The fused cell of cell_f.cu is the
  // route that removes these round trips for H = 128.)
  for (int g = 0; g < 2; ++g)
    if (launch_gemm_nt_tma(L.h, H, a->p.lin_w[g] + H, 2 * H, L.D + (size_t)g * H, 4 * H, k.rows, H, H, L.bsplit, st, gk)) return -1;
  G_LAUNCH(k_g_zr, "k_g_zr");
  if (launch_gemm_nt_tma(L.hR, H, a->p.lin_w[2] + H, 2 * H, L.D + 2 * H, 4 * H, k.rows, H, H, L.bsplit, st, gk)) return -1;
  k_g_c<<<cdiv(BN * (H / 4), 256), 256, 0, st>>>(k);
  REGT_LAUNCHED("k_g_c", st);
  return 0;
}

int cell_backward_g(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, T = a->T;
  const long long BN = (long long)a->B * a->N, rows = BN * T;
  GK k = make_gk(a, L);
  const GemmKind gk = gemm_kind(L);
  float* part = L.part;
  float* BhT = part;                       // [H][H]   scratch until the weight-gradient partials take over
  float* BzrT = part + (size_t)H * H;      // [H][2H]
  double* dpp = reinterpret_cast<double*>(part + (size_t)3 * H * H);   // [nb1][T] attention-gradient partials (fp64)
  k_g_pack_bt<<<cdiv(3ll * H * H, 256), 256, 0, st>>>(a->p.lin_w[0], a->p.lin_w[1], a->p.lin_w[2], H, BhT, BzrT);
  REGT_LAUNCHED("k_g_pack_bt", st);
  const int nb1 = (int)min(1024ll, (long long)cdiv(BN * (H / 4), 256));
  k.dp_part = dpp;
  k_g_b1<<<nb1, 256, 0, st>>>(k);
  REGT_LAUNCHED("k_g_b1", st);
  if (launch_f_sum_dpp(dpp, nb1, T, L.dprobs, st)) return -1;
  if (launch_gemm_nt_tma(L.D + 2 * H, 4 * H, BhT, H, L.Hn, H, rows, H, H, L.bsplit, st, gk)) return -1;            // dHR = Dh . B_h
  G_LAUNCH(k_g_b2, "k_g_b2");
  if (launch_gemm_nt_tma(L.D, 4 * H, BzrT, 2 * H, L.D + 3 * H, 4 * H, rows, H, 2 * H, L.bsplit, st, gk)) return -1;   // dhg
  G_LAUNCH(k_g_b3, "k_g_b3");
  // H x H weight gradients on the tensor cores (contraction over the rows)
  // ... and, in the SAME pass over D, the F-wide gradients and biases D^T . [S | X | 1] (second, 32-column operand:
  // the feature plane built in the forward).  H % 128 == 0: ONE launch over all four gate blocks of D (z | r against h,
  // h~ against h*R, h_pre against the feature plane only), split so that the grid fills the SMs once.
  const bool merged = H % 128 == 0;
  const int ctas_per_split = (4 * H / 128) * (H / 128);
  const int splits = merged ? (int)max(1ll, min((long long)min(WGRAD_SPLITS, cdiv(148, ctas_per_split)), rows / 512))
                            : (int)max(1ll, min((long long)WGRAD_SPLITS, rows / 512));
  float* pB = part;                                          // [splits][2H][H]  dB_z | dB_r
  float* pBh = pB + (size_t)splits * 2 * H * H;              // [splits][H][H]   dB_h
  float* pF = pBh + (size_t)splits * H * H;                  // [splits][4H][32] D^T Feat
  const long long fsplit = 4ll * H * 32;
  if (merged) {
    const int k0[3] = {0, 2 * H, 3 * H}, sb[3] = {0, 1, -1};
    float* cs[3] = {pB, pBh, nullptr};
    const float* bs[2] = {L.h, L.hR};
    const long long lds[2] = {H, H};
    if (launch_gemm_tn_tma(L.D, 4 * H, rows, 4 * H, 3, k0, sb, cs, bs, lds, H, splits, L.Feat, 32, pF, fsplit, st, 0, gk)) return -1;
  } else {
    if (launch_gemm_tn(L.D, 4 * H, L.h, H, pB, rows, 2 * H, H, splits, st, L.Feat, 32, pF, fsplit, 0, gk)) return -1;
    if (launch_gemm_tn(L.D + 2 * H, 4 * H, L.hR, H, pBh, rows, H, H, splits, st, L.Feat, 32, pF + (size_t)2 * H * 32, fsplit, 0, gk)) return -1;
    if (launch_gemm_tn(L.D + 3 * H, 4 * H, nullptr, 0, nullptr, rows, H, 0, splits, st, L.Feat, 32, pF + (size_t)3 * H * 32, fsplit, 0, gk)) return -1;
  }
  if (launch_reduce_splits(pB, L.dB, 2ll * H * H, splits, 0, st)) return -1;
  if (launch_reduce_splits(pBh, L.dB + (size_t)2 * H * H, (long long)H * H, splits, 0, st)) return -1;
  if (launch_fw_scatter(pF, splits, H, L, st)) return -1;
  if (a->mode != REGT_MODE_TGCN) {   // dM1[r]: per-region sums over the (node, region) segments
    if (launch_wgrad_m1(a, L, st)) return -1;
  }
  return launch_chain(a, L, st);
}

}  // namespace regt
