// Weight collapse (forward) and its chain rule (backward).  SURVEY Appendix B.
//
// The reference evaluates, per period, GCNConv(F->H) followed by Linear(2H->H) for each of
// the three gates (models/utils.py:168-184) and R ChebConv(F->H) followed by
// Linear(R*H->H) (models/RegionalTemporalGCN.py:136-142).  All of those are linear in the
// F-wide quantities S = A_hat X and U_r = L_hat_r X, so the H x H x F products are folded
// into the weights once per step:
//   P_g = A_g W_g,  c_g = A_g b_g + lb_g          with linear_g.weight = [A_g | B_g]
//   M0  = (sum_r L_r) W0,  M1[r] = L_r W1,  c0 = (sum_r L_r) b + b_lin
// These are tiny (H*H*F flops); they run as plain one-thread-per-output kernels with fp64
// accumulation so the collapse adds no rounding of its own.
//
// The parameters conv_w / cheb_w0 / cheb_w1 are [H, Fin] with the caller's Fin <= F (regt_args.F); everything collapsed
// is F wide.  Columns Fin..F-1 of the collapsed weights are written as zeros, and the chain rule reads the missing
// parameter columns as zeros and writes only the Fin real ones: the F-wide arithmetic of a zero-padded model.
#include "common.cuh"

namespace regt {

constexpr int F = REGT_F;

// element (m, f) of an [H, Fin] parameter, 0 for the padded columns f >= Fin
__device__ __forceinline__ float wcol(const float* w, int m, int f, int Fin) { return f < Fin ? w[(size_t)m * Fin + f] : 0.f; }

__global__ void k_lsum(const float* __restrict__ comb_w, int H, int R, float* __restrict__ Lsum) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * H) return;
  int j = i / H, m = i % H;
  double s = 0.0;
  for (int r = 0; r < R; ++r) s += comb_w[(size_t)j * R * H + (size_t)r * H + m];
  Lsum[i] = (float)s;
}

// flat output space: [0, n_w) packed gate weights, then biases, cheb pieces, probs.
// PG consecutive lanes share one output: each sums a slice of the H-long contraction in fp64, the
// slices are combined with a shuffle tree (the step waits on this kernel, so its latency -- a chain
// of H dependent loads from cold HBM per output in a one-thread-per-output form -- matters).
constexpr int PG = 8;
__global__ void __launch_bounds__(256) k_prep(regt_params p, int H, int Fin, int R, int T, int mode, const float* __restrict__ Lsum,
                                              float* __restrict__ Wzr, float* __restrict__ Wc, float* __restrict__ czr,
                                              float* __restrict__ cc, float* __restrict__ M0t, float* __restrict__ M1t,
                                              float* __restrict__ c0, float* __restrict__ probs) {
  const long long nW = (long long)3 * (F + H) * H;  // gate weights
  const long long nC = 3 * H;                       // gate biases
  const long long nM0 = (long long)F * H, nM1 = (long long)R * F * H, nc0 = H;
  const long long gt = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long i = gt / PG;
  const int sub = (int)(gt % PG), m0 = sub * (H / PG), m1 = m0 + H / PG;   // H % 8 == 0 (validated)
  double s = 0.0;       // this lane's slice of the contraction (or the whole value for copies, lane 0)
  float* dst = nullptr;
  if (i < nW) {
    int g = (int)(i / ((F + H) * H));
    int rem = (int)(i % ((F + H) * H));
    int k = rem / H, j = rem % H;  // j fastest: coalesced writes
    if (k < Fin) {
      const float* A = p.lin_w[g] + (size_t)j * 2 * H;
      const float* W = p.conv_w[g];
      for (int m = m0; m < m1; ++m) s += (double)__ldg(A + m) * (double)__ldg(W + m * Fin + k);
    } else if (k >= F && sub == 0) {   // k in [Fin, F): zero column
      s = p.lin_w[g][(size_t)j * 2 * H + H + (k - F)];
    }
    dst = (g < 2) ? Wzr + (size_t)k * 2 * H + g * H + j : Wc + (size_t)k * H + j;
  } else if ((i -= nW) < nC) {
    int g = (int)(i / H), j = (int)(i % H);
    if (sub == 0) s = p.lin_b[g][j];
    const float* A = p.lin_w[g] + (size_t)j * 2 * H;
    for (int m = m0; m < m1; ++m) s += (double)__ldg(A + m) * (double)__ldg(p.conv_b[g] + m);
    dst = (g < 2) ? czr + g * H + j : cc + j;
  } else if (mode == REGT_MODE_TGCN) {  // no Chebyshev branch: only probs (T == 1 -> 1.0)
    i -= nC;
    if (i == 0 && sub == 0) {
      float mx = -INFINITY;
      for (int t = 0; t < T; ++t) mx = fmaxf(mx, p.attention ? p.attention[t] : 0.f);
      double den = 0.0;
      for (int t = 0; t < T; ++t) den += exp((double)(p.attention ? p.attention[t] : 0.f) - mx);
      for (int t = 0; t < T; ++t) probs[t] = (float)(exp((double)(p.attention ? p.attention[t] : 0.f) - mx) / den);
    }
  } else if ((i -= nC) < nM0) {
    int f = (int)(i / H), j = (int)(i % H);
    if (f >= Fin) {   // padded column: 0
    } else if (mode == REGT_MODE_REGIONAL) {
      for (int m = m0; m < m1; ++m) s += (double)__ldg(Lsum + (size_t)j * H + m) * (double)__ldg(p.cheb_w0 + m * Fin + f);
    } else if (sub == 0) {
      s = p.cheb_w0[j * Fin + f];
    }
    dst = M0t + i;
  } else if ((i -= nM0) < nM1) {
    int r = (int)(i / (F * H));
    int rem = (int)(i % (F * H));
    int f = rem / H, j = rem % H;
    if (f >= Fin) {   // padded column: 0
    } else if (mode == REGT_MODE_REGIONAL) {
      const float* L = p.comb_w + (size_t)j * R * H + (size_t)r * H;
      for (int m = m0; m < m1; ++m) s += (double)__ldg(L + m) * (double)__ldg(p.cheb_w1 + m * Fin + f);
    } else if (sub == 0) {
      s = p.cheb_w1[j * Fin + f];
    }
    dst = M1t + i;
  } else if ((i -= nM1) < nc0) {
    int j = (int)i;
    if (mode == REGT_MODE_REGIONAL) {
      if (sub == 0) s = p.comb_b[j];
      for (int m = m0; m < m1; ++m) s += (double)__ldg(Lsum + (size_t)j * H + m) * (double)__ldg(p.cheb_b + m);
    } else if (sub == 0) {
      s = p.cheb_b[j];
    }
    dst = c0 + j;
  } else if ((i -= nc0) == 0 && sub == 0) {
    attention_softmax(p.attention, T, probs);   // softmax over the T learned scalars (models/RegionalTemporalGCN.py:134)
  }
  // all 32 lanes reach this point: combine the PG slices (fixed tree: deterministic)
#pragma unroll
  for (int d = PG / 2; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if (dst && sub == 0) *dst = (float)s;
}

int launch_prep(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, R = a->plan.R;
  if (a->mode == REGT_MODE_REGIONAL) {
    k_lsum<<<cdiv((long long)H * H, 256), 256, 0, st>>>(a->p.comb_w, H, R, L.Lsum);
    REGT_LAUNCHED("k_lsum", st);
  }
  long long n = (long long)3 * (F + H) * H + 3 * H + (long long)F * H + (long long)R * F * H + H + 1;
  k_prep<<<cdiv(n * PG, 256), 256, 0, st>>>(a->p, H, feat_in(a), R, a->T, a->mode, L.Lsum, L.Wzr, L.Wc, L.czr, L.cc, L.M0t, L.M1t, L.c0,
                                      L.probs);
  REGT_LAUNCHED("k_prep", st);
  return 0;
}

// ---------------------------------------------------------------------------------------
// chain rule from collapsed-weight gradients to the reference parameters
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void put(float* dst, size_t i, double v, int acc) {
  if (!dst) return;
  dst[i] = acc ? dst[i] + (float)v : (float)v;
}

__global__ void k_chain(regt_params p, regt_params g, int H, int Fin, int R, int T, int mode, int acc,
                        const float* __restrict__ Lsum, const float* __restrict__ probs,
                        const float* __restrict__ dB, const float* __restrict__ dP, const float* __restrict__ dcg,
                        const float* __restrict__ dM0, const float* __restrict__ dM1, const float* __restrict__ dc0,
                        const float* __restrict__ dprobs) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long nLW = (long long)3 * H * 2 * H, nLB = 3 * H, nCW = (long long)3 * H * Fin, nCB = 3 * H;
  if (i < nLW) {  // linear_g.weight [H,2H] = [dA_g | dB_g]
    int gI = (int)(i / ((long long)H * 2 * H));
    int rem = (int)(i % ((long long)H * 2 * H));
    int j = rem / (2 * H), c = rem % (2 * H);
    double v;
    if (c < H) {
      v = (double)dcg[gI * H + j] * (double)p.conv_b[gI][c];
      for (int f = 0; f < F; ++f) v += (double)dP[((size_t)gI * H + j) * F + f] * (double)wcol(p.conv_w[gI], c, f, Fin);
    } else {
      v = dB[((size_t)gI * H + j) * H + (c - H)];
    }
    put(g.lin_w[gI], (size_t)j * 2 * H + c, v, acc);
    return;
  }
  i -= nLW;
  if (i < nLB) {
    int gI = (int)(i / H), j = (int)(i % H);
    put(g.lin_b[gI], j, dcg[gI * H + j], acc);
    return;
  }
  i -= nLB;
  if (i < nCW) {  // conv_g.lin.weight [H,Fin] = A_g^T dP_g (the real columns)
    int gI = (int)(i / (H * Fin));
    int rem = (int)(i % (H * Fin));
    int m = rem / Fin, f = rem % Fin;
    double v = 0.0;
    for (int j = 0; j < H; ++j) v += (double)p.lin_w[gI][(size_t)j * 2 * H + m] * (double)dP[((size_t)gI * H + j) * F + f];
    put(g.conv_w[gI], (size_t)m * Fin + f, v, acc);
    return;
  }
  i -= nCW;
  if (i < nCB) {
    int gI = (int)(i / H), m = (int)(i % H);
    double v = 0.0;
    for (int j = 0; j < H; ++j) v += (double)p.lin_w[gI][(size_t)j * 2 * H + m] * (double)dcg[gI * H + j];
    put(g.conv_b[gI], m, v, acc);
    return;
  }
  i -= nCB;
  if (i < T) {  // softmax backward
    if (mode == REGT_MODE_TGCN || !g.attention) return;
    int t = (int)i;
    double dot = 0.0;
    for (int s = 0; s < T; ++s) dot += (double)probs[s] * (double)dprobs[s];
    put(g.attention, t, (double)probs[t] * ((double)dprobs[t] - dot), acc);
    return;
  }
  i -= T;
  if (mode == REGT_MODE_TGCN) return;
  const long long nW0 = (long long)H * Fin;
  if (i < 2 * nW0) {  // cheb lins.0 / lins.1 weights [H,Fin]
    int which = (int)(i / nW0);
    int rem = (int)(i % nW0);
    int m = rem / Fin, f = rem % Fin;
    double v = 0.0;
    if (mode == REGT_MODE_REGIONAL) {
      if (which == 0) {
        for (int j = 0; j < H; ++j) v += (double)Lsum[(size_t)j * H + m] * (double)dM0[(size_t)j * F + f];
      } else {
        return;   // R*H-long contraction: one block per output (k_chain_w1)
      }
    } else {
      v = which == 0 ? dM0[(size_t)m * F + f] : dM1[(size_t)m * F + f];
    }
    put(which == 0 ? g.cheb_w0 : g.cheb_w1, (size_t)m * Fin + f, v, acc);
    return;
  }
  i -= 2 * nW0;
  if (i < H) {  // cheb bias
    int m = (int)i;
    double v = 0.0;
    if (mode == REGT_MODE_REGIONAL) {
      for (int j = 0; j < H; ++j) v += (double)Lsum[(size_t)j * H + m] * (double)dc0[j];
    } else {
      v = dc0[m];
    }
    put(g.cheb_b, m, v, acc);
    return;
  }
  i -= H;
  if (mode != REGT_MODE_REGIONAL) return;
  if (i < H) {
    put(g.comb_b, (size_t)i, dc0[i], acc);
    return;
  }
  i -= H;
  const long long nL = (long long)H * R * H;
  if (i < nL) {  // linear.weight [H, R*H]: dL_r = dM0 W0^T + dM1[r] W1^T + dc0 b^T
    int j = (int)(i / ((long long)R * H));
    int rem = (int)(i % ((long long)R * H));
    int r = rem / H, m = rem % H;
    double v = (double)dc0[j] * (double)p.cheb_b[m];
    for (int f = 0; f < F; ++f) {
      v += (double)dM0[(size_t)j * F + f] * (double)wcol(p.cheb_w0, m, f, Fin);
      v += (double)dM1[((size_t)r * H + j) * F + f] * (double)wcol(p.cheb_w1, m, f, Fin);
    }
    put(g.comb_w, (size_t)i, v, acc);
  }
}

// cheb lins.1 weight of the regional model: d W1[m][f] = sum_r sum_j L_r[j][m] * dM1[r][j][f]  (R*H terms per output)
__global__ void __launch_bounds__(256) k_chain_w1(const float* __restrict__ comb_w, const float* __restrict__ dM1, int H, int Fin,
                                                  int R, int acc, float* __restrict__ g_w1) {
  __shared__ double red[256];
  const int m = blockIdx.x / Fin, f = blockIdx.x % Fin;
  double v = 0.0;
  for (int i = threadIdx.x; i < R * H; i += 256) {   // i = r*H + j ; fixed strided order, then a fixed tree
    const int r = i / H, j = i - r * H;
    v += (double)__ldg(comb_w + (size_t)j * R * H + (size_t)r * H + m) * (double)__ldg(dM1 + ((size_t)r * H + j) * F + f);
  }
  red[threadIdx.x] = v;
  __syncthreads();
  for (int d = 128; d > 0; d >>= 1) {
    if (threadIdx.x < d) red[threadIdx.x] += red[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0 && g_w1) g_w1[(size_t)m * Fin + f] = acc ? g_w1[(size_t)m * Fin + f] + (float)red[0] : (float)red[0];
}

int launch_chain(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, R = a->plan.R, Fin = feat_in(a);
  long long n = (long long)3 * H * 2 * H + 3 * H + (long long)3 * H * Fin + 3 * H + a->T + 2ll * H * Fin + H + H +
                (long long)H * R * H;
  k_chain<<<cdiv(n, 256), 256, 0, st>>>(a->p, a->g, H, Fin, R, a->T, a->mode, a->accumulate, L.Lsum, L.probs, L.dB, L.dP,
                                       L.dcg, L.dM0, L.dM1, L.dc0, L.dprobs);
  REGT_LAUNCHED("k_chain", st);
  if (a->mode == REGT_MODE_REGIONAL) {
    k_chain_w1<<<H * Fin, 256, 0, st>>>(a->p.comb_w, L.dM1, H, Fin, R, a->accumulate, a->g.cheb_w1);
    REGT_LAUNCHED("k_chain_w1", st);
  }
  return 0;
}

}  // namespace regt
