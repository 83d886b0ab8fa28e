// fp32 (REGT_PREC_FP32) kernels of the regional temporal GCN cell: forward and backward.
//
// Row index of every [rows, H] plane: row = (b*N + n)*T + t  (periods are independent --
// SURVEY fact 5 -- so T folds into the row dimension).  Per row the cell is
//   h   = act( X_t M0 + sum_seg U_seg,t M1[r_seg] + c0 )            (regional combine, collapsed)
//   Z,R = sigmoid( [S_t | h] Wzr + czr )                            (models/utils.py:168-178)
//   H~  = tanh( [S_t | h*R] Wc + cc )                               (models/utils.py:180-184)
//   H'  = Z*h + (1-Z)*H~                                            (models/utils.py:186-188)
//   out_hidden[b,n] = sum_t softmax(attention)[t] * H'              (RegionalTemporalGCN.py:134,146)
// with S = A_hat X, U = L_hat_r X the F-wide SpMM results (spmm.cu).
#include "gemm_simt.cuh"

namespace regt {

constexpr int F = REGT_F;

struct CellK {
  int rows, N, xN, T, H, nseg, mode;   // xN: node rows per snapshot of x (>= N: halo rows of a region shard)
  const float *x, *S, *U, *h_ext;
  const int32_t *seg_ptr, *seg_reg;
  const float *M0t, *M1t, *c0, *Wzr, *Wc, *czr, *cc, *probs;
  float *h, *Z, *Rg, *Hc, *hR, *Hn;
  // backward
  const float* G;       // [B*N][H]
  const float* lin_w[3];  // linear_{z,r,h}.weight [H][2H]; B_g = columns H..2H-1
  float* D;             // [rows][4H]
  float* d_h_ext;
};

__device__ __forceinline__ void st4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int TM>
__global__ void __launch_bounds__(TM * 4) k_cell_fwd(CellK a) {
  constexpr int NT = TM * 4;
  extern __shared__ __align__(16) float smem[];
  const int H = a.H, T = a.T, lda = F + H + 1;
  float* A1s = smem;             // [TM][lda]  (S_t | h)
  float* A2s = A1s + TM * lda;   // [TM][lda]  (S_t | h*R)
  float* Ws = A2s + TM * lda;    // [KT*TN]  (16-byte aligned: TM*lda*2 floats is a multiple of 4)
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const long long row0 = (long long)blockIdx.x * TM;

  // ---- prologue: h (regional combine on F-wide features) and S into shared memory ----
  for (int idx = tid; idx < TM * H; idx += NT) {
    const int rl = idx / H, j = idx - rl * H;
    const long long row = row0 + rl;
    float hv = 0.f;
    if (row < a.rows) {
      if (a.mode == REGT_MODE_TGCN) {
        hv = a.h_ext ? a.h_ext[row * H + j] : 0.f;
      } else {
        const long long q = row / T;
        const int t = (int)(row - q * T);
        const int b = (int)(q / a.N), n = (int)(q - (long long)b * a.N);
        const float* xr = a.x + ((size_t)b * a.xN + n) * F * T + t;
        float acc = a.c0[j];
#pragma unroll
        for (int f = 0; f < F; ++f) acc = fmaf(__ldg(xr + f * T), __ldg(a.M0t + f * H + j), acc);
        for (int s = a.seg_ptr[n]; s < a.seg_ptr[n + 1]; ++s) {
          const float* ur = a.U + ((size_t)b * a.nseg + s) * F * T + t;
          const float* m = a.M1t + (size_t)a.seg_reg[s] * F * H + j;
#pragma unroll
          for (int f = 0; f < F; ++f) acc = fmaf(__ldg(ur + f * T), __ldg(m + f * H), acc);
        }
        hv = (a.mode == REGT_MODE_REGIONAL) ? (acc > 0.f ? acc : 0.01f * acc) : acc;  // F.leaky_relu
      }
      a.h[row * H + j] = hv;
    }
    A1s[rl * lda + F + j] = hv;
  }
  for (int idx = tid; idx < TM * F; idx += NT) {
    const int rl = idx / F, f = idx - rl * F;
    const long long row = row0 + rl;
    float v = 0.f;
    if (row < a.rows) {
      const long long q = row / T;
      const int t = (int)(row - q * T);
      v = __ldg(a.S + q * F * T + f * T + t);
    }
    A1s[rl * lda + f] = v;
    A2s[rl * lda + f] = v;
  }
  __syncthreads();

  // ---- update / reset gates:  [S|h] Wzr ----
  for (int n0 = 0; n0 < 2 * H; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(A1s, lda, F + H, a.Wzr, 2 * H, n0, 2 * H, Ws, acc, ty, tx);
    const int n = n0 + tx * 4;
    if (n < 2 * H) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = ty * 4 + i;
        const long long row = row0 + rl;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = sigmoidf_(acc[i][j] + __ldg(a.czr + n + j));
        if (n < H) {
          if (row < a.rows) st4(a.Z + row * H + n, v[0], v[1], v[2], v[3]);
        } else {
          const int nn = n - H;
          float hr[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            hr[j] = A1s[rl * lda + F + nn + j] * v[j];
            A2s[rl * lda + F + nn + j] = hr[j];
          }
          if (row < a.rows) {
            st4(a.Rg + row * H + nn, v[0], v[1], v[2], v[3]);
            st4(a.hR + row * H + nn, hr[0], hr[1], hr[2], hr[3]);
          }
        }
      }
    }
  }
  __syncthreads();

  // ---- candidate + blend:  [S|h*R] Wc ----
  for (int n0 = 0; n0 < H; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(A2s, lda, F + H, a.Wc, H, n0, H, Ws, acc, ty, tx);
    const int n = n0 + tx * 4;
    if (n < H) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = ty * 4 + i;
        const long long row = row0 + rl;
        if (row >= a.rows) continue;
        const float4 z4 = *reinterpret_cast<const float4*>(a.Z + row * H + n);  // written above by this thread
        const float z[4] = {z4.x, z4.y, z4.z, z4.w};
        float hc[4], hn[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          hc[j] = tanhf(acc[i][j] + __ldg(a.cc + n + j));
          const float hv = A1s[rl * lda + F + n + j];
          hn[j] = z[j] * hv + (1.0f - z[j]) * hc[j];
        }
        st4(a.Hc + row * H + n, hc[0], hc[1], hc[2], hc[3]);
        st4(a.Hn + row * H + n, hn[0], hn[1], hn[2], hn[3]);
      }
    }
  }
}

// K3: period attention  out_hidden[q] = sum_t probs[t] * H'[q,t]
__global__ void k_attn_accum(const float* __restrict__ Hn, const float* __restrict__ probs, int T, int H,
                             long long BN, float* __restrict__ out_hidden) {
  const int H4 = H / 4;
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= BN * H4) return;
  const long long q = i / H4;
  const int j4 = (int)(i - q * H4);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int t = 0; t < T; ++t) {
    const float p = __ldg(probs + t);
    const float4 v = __ldg(reinterpret_cast<const float4*>(Hn + (q * T + t) * H) + j4);
    acc.x = fmaf(p, v.x, acc.x);
    acc.y = fmaf(p, v.y, acc.y);
    acc.z = fmaf(p, v.z, acc.z);
    acc.w = fmaf(p, v.w, acc.w);
  }
  reinterpret_cast<float4*>(out_hidden + q * H)[j4] = acc;
}

// ------------------------------------------------------------------------------------------
// backward: elementwise GRU/attention chain + the two data-gradient contractions
// ------------------------------------------------------------------------------------------
template <int TM>
__global__ void __launch_bounds__(TM * 4) k_cell_bwd(CellK a) {
  constexpr int NT = TM * 4;
  extern __shared__ __align__(16) float smem[];
  const int H = a.H, T = a.T, ldh = H + 1;
  float* Dz = smem;            // d pre_z
  float* Dr = Dz + TM * ldh;   // d pre_r
  float* Dh = Dr + TM * ldh;   // d pre_h
  float* dhs = Dh + TM * ldh;  // running d h
  float* Ws = dhs + TM * ldh + ((4 - ((4 * TM * ldh) & 3)) & 3);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const long long row0 = (long long)blockIdx.x * TM;

  for (int idx = tid; idx < TM * H; idx += NT) {
    const int rl = idx / H, j = idx - rl * H;
    const long long row = row0 + rl;
    float dz = 0.f, dh_ = 0.f, dhc = 0.f;
    if (row < a.rows) {
      const long long q = row / T;
      const int t = (int)(row - q * T);
      const float g = __ldg(a.probs + t) * __ldg(a.G + q * H + j);  // dH' = probs[t] * dH_accum
      const float hv = a.h[row * H + j], z = a.Z[row * H + j], hc = a.Hc[row * H + j];
      const float dZ = g * (hv - hc);
      const float dHc = g * (1.0f - z);
      dh_ = g * z;
      dhc = dHc * (1.0f - hc * hc);
      dz = dZ * z * (1.0f - z);
    }
    Dz[rl * ldh + j] = dz;
    Dh[rl * ldh + j] = dhc;
    dhs[rl * ldh + j] = dh_;
  }
  // d(h*R) = d pre_h . B_h ;  B_h[n][k] = linear_h.weight[n][H+k]
  for (int n0 = 0; n0 < H; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(Dh, ldh, H, a.lin_w[2] + H, 2 * H, n0, H, Ws, acc, ty, tx);
    const int k = n0 + tx * 4;
    if (k < H) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = ty * 4 + i;
        const long long row = row0 + rl;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float dr = 0.f;
          if (row < a.rows) {
            const float hv = a.h[row * H + k + j], r = a.Rg[row * H + k + j];
            const float dHR = acc[i][j];
            dhs[rl * ldh + k + j] += dHR * r;
            dr = dHR * hv * r * (1.0f - r);
          }
          Dr[rl * ldh + k + j] = dr;
        }
      }
    }
  }
  // d h += d pre_z . B_z + d pre_r . B_r ; then through the regional combine's activation
  for (int n0 = 0; n0 < H; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(Dz, ldh, H, a.lin_w[0] + H, 2 * H, n0, H, Ws, acc, ty, tx);
    tile_gemm<NT>(Dr, ldh, H, a.lin_w[1] + H, 2 * H, n0, H, Ws, acc, ty, tx);
    const int k = n0 + tx * 4;
    if (k < H) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = ty * 4 + i;
        const long long row = row0 + rl;
        if (row >= a.rows) continue;
        float dpre[4], vz[4], vr[4], vh[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float dh_total = dhs[rl * ldh + k + j] + acc[i][j];
          if (a.mode == REGT_MODE_TGCN) {
            if (a.d_h_ext) a.d_h_ext[row * H + k + j] = dh_total;
            dpre[j] = 0.f;
          } else if (a.mode == REGT_MODE_REGIONAL) {
            dpre[j] = dh_total * (a.h[row * H + k + j] > 0.f ? 1.0f : 0.01f);
          } else {
            dpre[j] = dh_total;
          }
          vz[j] = Dz[rl * ldh + k + j];
          vr[j] = Dr[rl * ldh + k + j];
          vh[j] = Dh[rl * ldh + k + j];
        }
        float* d = a.D + row * 4 * H + k;
        st4(d, vz[0], vz[1], vz[2], vz[3]);
        st4(d + H, vr[0], vr[1], vr[2], vr[3]);
        st4(d + 2 * H, vh[0], vh[1], vh[2], vh[3]);
        st4(d + 3 * H, dpre[0], dpre[1], dpre[2], dpre[3]);
      }
    }
  }
}

// d probs[t] = sum_{q,j} G[q][j] * H'[q,t][j]   ->  part[blk][t]
__global__ void __launch_bounds__(256) k_dprobs(const float* __restrict__ G, const float* __restrict__ Hn, int T, int H,
                                                long long BN, float* __restrict__ part) {
  __shared__ float red[32];
  const long long total = BN * H;
  for (int t = 0; t < T; ++t) {
    float s = 0.f;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long q = i / H;
      const int j = (int)(i - q * H);
      s = fmaf(__ldg(G + i), __ldg(Hn + (q * T + t) * H + j), s);
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[(size_t)blockIdx.x * T + t] = s;
  }
}

// ---- F-wide weight gradients: dP_g = D_g^T S, dM0 = D_3^T X, biases = column sums ----------
// thread c owns one column of D; part[split][c][F+1]
__global__ void __launch_bounds__(128) k_wgrad_skinny(const float* __restrict__ D, const float* __restrict__ S,
                                                      const float* __restrict__ x, int N, int xN, int H, int T,
                                                      long long rows, int ncol, long long chunk,
                                                      float* __restrict__ part) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  const long long r0 = blockIdx.y * chunk, r1 = min(rows, r0 + chunk);
  float acc[F + 1];
#pragma unroll
  for (int f = 0; f <= F; ++f) acc[f] = 0.f;
  if (c < ncol) {
    const bool from_x = c >= 3 * H;
    for (long long r = r0; r < r1; ++r) {
      const float d = __ldg(D + r * 4 * H + c);
      long long q = r / T;
      const int t = (int)(r - q * T);
      if (from_x && xN != N) q = (q / N) * xN + q % N;   // x carries halo rows after the N owned ones
      const float* fr = (from_x ? x : S) + q * F * T + t;
#pragma unroll
      for (int f = 0; f < F; ++f) acc[f] = fmaf(d, __ldg(fr + f * T), acc[f]);
      acc[F] += d;
    }
    float* o = part + ((size_t)blockIdx.y * ncol + c) * (F + 1);
#pragma unroll
    for (int f = 0; f <= F; ++f) o[f] = acc[f];
  }
}
__global__ void k_skinny_reduce(const float* __restrict__ part, int splits, int H, int ncol, float* __restrict__ dP,
                                float* __restrict__ dcg, float* __restrict__ dM0, float* __restrict__ dc0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncol * (F + 1)) return;
  const int c = i / (F + 1), f = i - c * (F + 1);
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += part[((size_t)sp * ncol + c) * (F + 1) + f];
  if (c < 3 * H) {
    if (f < F) dP[(size_t)c * F + f] = s; else dcg[c] = s;
  } else {
    const int n = c - 3 * H;
    if (f < F) dM0[(size_t)n * F + f] = s; else dc0[n] = s;
  }
}

// dM1[r] = sum over the (node, region r) segments of dhp^T U          (models/RegionalTemporalGCN.py:136-141 backward)
// Work items = (segment, snapshot) pairs in region-sorted order (rseg_list).  A region is cut into chunks of at most
// `per` items; chunk_ptr[r] = number of chunks before region r (k_m1_chunks), so EMPTY regions -- every list a region
// shard does not own -- cost nothing and the grid follows the work, not R.  A block owns one chunk: its warps stride
// over the chunk's items, a lane owns four gate columns (one 128-bit load per period, all T periods in flight), the
// item's U row [F][T] is a warp-uniform broadcast.  part[chunk][H][F]; k_m1_reduce sums a region's chunks in order.
constexpr int M1_TARGET_CHUNKS = 2048;
__global__ void k_m1_chunks(const int32_t* __restrict__ rseg_ptr, int R, int B, int per, int32_t* __restrict__ chunk_ptr) {
  __shared__ int part_sum[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int per_thr = (R + nt - 1) / nt;
  const int r0 = min(R, tid * per_thr), r1 = min(R, r0 + per_thr);
  int s = 0;
  for (int r = r0; r < r1; ++r) {
    const long long items = (long long)(rseg_ptr[r + 1] - rseg_ptr[r]) * B;
    s += (int)((items + per - 1) / per);
  }
  part_sum[tid] = s;
  __syncthreads();
  if (tid == 0) {   // exclusive scan of <= 1024 slice sums
    int run = 0;
    for (int i = 0; i < nt; ++i) {
      const int v = part_sum[i];
      part_sum[i] = run;
      run += v;
    }
    chunk_ptr[R] = run;
  }
  __syncthreads();
  int run = part_sum[tid];
  for (int r = r0; r < r1; ++r) {
    chunk_ptr[r] = run;
    const long long items = (long long)(rseg_ptr[r + 1] - rseg_ptr[r]) * B;
    run += (int)((items + per - 1) / per);
  }
}

// element strides of the two operands (two plane layouts feed this kernel):
//   dhp(b, node, t)[n] = dhp[(b*N + node) * d_qs + t * d_ts + n]      U(b, seg, f, t) = U[b * u_bs + seg * u_ss + f * u_fs + t * u_ts]
//   row = (b*N+n)*T + t planes (cell.cu, cell_g.cu): d_qs = T*ldd, d_ts = ldd ; U [B][nseg][F][T]: u_bs = nseg*F*T, u_ss = F*T, u_fs = T, u_ts = 1
//   period-major planes (cell_f.cu), row = t*BNp + q:  d_qs = ldd, d_ts = BNp*ldd ; Ut [T][B*nseg][F]: u_bs = nseg*F, u_ss = F, u_fs = 1, u_ts = B*nseg*F
struct M1Strides {
  long long d_qs, d_ts, u_bs, u_ss, u_fs, u_ts;
};
template <int TT>   // TT = periods held in flight per pass (T is processed in groups of TT)
__global__ void __launch_bounds__(128) k_wgrad_m1(const float* __restrict__ dhp, M1Strides sd, const float* __restrict__ U,
                                                  const int32_t* __restrict__ rseg_ptr, const int32_t* __restrict__ rseg_list,
                                                  const int32_t* __restrict__ seg_node, const int32_t* __restrict__ chunk_ptr,
                                                  int B, int N, int T, int H, int R, int nseg, int per,
                                                  float* __restrict__ part) {
  __shared__ float red[3][32][4 * F + 1];
  const int c = blockIdx.x;
  if (c >= chunk_ptr[R]) return;
  int lo = 0, hi = R;             // region of this chunk: largest r with chunk_ptr[r] <= c (empty regions share a value)
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (chunk_ptr[mid] <= c) lo = mid; else hi = mid;
  }
  const int r = lo;
  const int s0 = rseg_ptr[r];
  const long long items = (long long)(rseg_ptr[r + 1] - s0) * B;
  const long long i0 = (long long)(c - chunk_ptr[r]) * per, i1 = min(items, i0 + per);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.y * 128 + lane * 4;
  const bool n_ok = n < H;
  float acc[4][F];
#pragma unroll
  for (int e = 0; e < 4; ++e)
#pragma unroll
    for (int f = 0; f < F; ++f) acc[e][f] = 0.f;
  for (long long i = i0 + warp; i < i1; i += 4) {
    const int s = rseg_list[s0 + (int)(i / B)];
    const int b = (int)(i % B);
    const int node = seg_node[s];
    const float* ur = U + (size_t)b * sd.u_bs + (size_t)s * sd.u_ss;
    const float* dr = dhp + ((size_t)b * N + node) * sd.d_qs + n;
    for (int t0 = 0; t0 < T; t0 += TT) {
      float4 d[TT];
#pragma unroll
      for (int k = 0; k < TT; ++k)
        d[k] = (n_ok && t0 + k < T) ? __ldg(reinterpret_cast<const float4*>(dr + (size_t)(t0 + k) * sd.d_ts)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int f = 0; f < F; ++f) {
#pragma unroll
        for (int k = 0; k < TT; ++k) {
          const float u = (t0 + k < T) ? __ldg(ur + f * sd.u_fs + (t0 + k) * sd.u_ts) : 0.f;
          acc[0][f] = fmaf(d[k].x, u, acc[0][f]);
          acc[1][f] = fmaf(d[k].y, u, acc[1][f]);
          acc[2][f] = fmaf(d[k].z, u, acc[2][f]);
          acc[3][f] = fmaf(d[k].w, u, acc[3][f]);
        }
      }
    }
  }
  // warps 1..3 hand their sums to warp 0 (fixed order -> deterministic)
  if (warp > 0) {
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
      for (int f = 0; f < F; ++f) red[warp - 1][lane][e * F + f] = acc[e][f];
  }
  __syncthreads();
  if (warp == 0 && n_ok) {
#pragma unroll
    for (int w = 0; w < 3; ++w)
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int f = 0; f < F; ++f) acc[e][f] += red[w][lane][e * F + f];
    float* o = part + ((size_t)c * H + n) * F;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      *reinterpret_cast<float4*>(o + e * F) = make_float4(acc[e][0], acc[e][1], acc[e][2], acc[e][3]);
      *reinterpret_cast<float4*>(o + e * F + 4) = make_float4(acc[e][4], acc[e][5], acc[e][6], acc[e][7]);
    }
  }
}
// period-major variant (planes of cell_f.cu: row = t*BNp + q, Ut [T][B*nseg][F]): the F values of an item's period are two
// warp-uniform 128-bit loads (the strided layout above needs 8 scalar loads per period), TT periods in flight
template <int TT>
__global__ void __launch_bounds__(128) k_wgrad_m1_pm(const float* __restrict__ dhp, long long ldd, long long d_ts,
                                                     const float* __restrict__ Ut, long long u_ts,
                                                     const int32_t* __restrict__ rseg_ptr, const int32_t* __restrict__ rseg_list,
                                                     const int32_t* __restrict__ seg_node, const int32_t* __restrict__ chunk_ptr,
                                                     int B, int N, int T, int H, int R, int nseg, int per, float* __restrict__ part) {
  __shared__ float red[3][32][4 * F + 1];
  const int c = blockIdx.x;
  if (c >= chunk_ptr[R]) return;
  int lo = 0, hi = R;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (chunk_ptr[mid] <= c) lo = mid; else hi = mid;
  }
  const int r = lo;
  const int s0 = rseg_ptr[r];
  const long long items = (long long)(rseg_ptr[r + 1] - s0) * B;
  const long long i0 = (long long)(c - chunk_ptr[r]) * per, i1 = min(items, i0 + per);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.y * 128 + lane * 4;
  const bool n_ok = n < H;
  float acc[4][F];
#pragma unroll
  for (int e = 0; e < 4; ++e)
#pragma unroll
    for (int f = 0; f < F; ++f) acc[e][f] = 0.f;
  for (long long i = i0 + warp; i < i1; i += 4) {
    const int s = rseg_list[s0 + (int)(i / B)];
    const int b = (int)(i % B);
    const int node = seg_node[s];
    const float4* ur = reinterpret_cast<const float4*>(Ut + ((size_t)b * nseg + s) * F);
    const float* dr = dhp + ((size_t)b * N + node) * ldd + n;
    for (int t0 = 0; t0 < T; t0 += TT) {
      float4 d[TT], ua[TT], ub[TT];
#pragma unroll
      for (int k = 0; k < TT; ++k) {
        const bool ok = t0 + k < T;
        d[k] = (n_ok && ok) ? __ldg(reinterpret_cast<const float4*>(dr + (size_t)(t0 + k) * d_ts)) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4* up = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ur) + (size_t)(ok ? t0 + k : 0) * u_ts);
        ua[k] = __ldg(up);
        ub[k] = __ldg(up + 1);
      }
#pragma unroll
      for (int k = 0; k < TT; ++k) {
        const float u[F] = {ua[k].x, ua[k].y, ua[k].z, ua[k].w, ub[k].x, ub[k].y, ub[k].z, ub[k].w};
#pragma unroll
        for (int f = 0; f < F; ++f) {
          acc[0][f] = fmaf(d[k].x, u[f], acc[0][f]);
          acc[1][f] = fmaf(d[k].y, u[f], acc[1][f]);
          acc[2][f] = fmaf(d[k].z, u[f], acc[2][f]);
          acc[3][f] = fmaf(d[k].w, u[f], acc[3][f]);
        }
      }
    }
  }
  if (warp > 0) {
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
      for (int f = 0; f < F; ++f) red[warp - 1][lane][e * F + f] = acc[e][f];
  }
  __syncthreads();
  if (warp == 0 && n_ok) {
#pragma unroll
    for (int w = 0; w < 3; ++w)
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int f = 0; f < F; ++f) acc[e][f] += red[w][lane][e * F + f];
    float* o = part + ((size_t)c * H + n) * F;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      *reinterpret_cast<float4*>(o + e * F) = make_float4(acc[e][0], acc[e][1], acc[e][2], acc[e][3]);
      *reinterpret_cast<float4*>(o + e * F + 4) = make_float4(acc[e][4], acc[e][5], acc[e][6], acc[e][7]);
    }
  }
}
// transposed variant (planes of cell_f.cu): dhp lives in D^T tiles [tp][4 row quarters][4H][32 rows] (tp = t * nqt + qt), Ut is period
// major.  Lanes run along the SEGMENTS of a region (= consecutive nodes = consecutive rows of a tile: 128-byte lines of every
// D^T column), a warp owns NPW gate columns, a thread keeps NPW x F running sums over all its rows and the 32 row lanes
// are summed once per chunk (butterfly, fixed order).  Chunk = (region, group of bper snapshots): part[chunk][H][F].
template <int NPW>
__global__ void __launch_bounds__(512) k_wgrad_m1_kt(const float* __restrict__ DT, int Ktot, int col0, const float* __restrict__ Ut,
                                                     const int32_t* __restrict__ rseg_ptr, const int32_t* __restrict__ rseg_list,
                                                     const int32_t* __restrict__ seg_node, int B, int N, int T, int nqt, int nseg,
                                                     int nbg, int bper, int H, float* __restrict__ part) {
  const int c = blockIdx.x, r = c / nbg, bg = c - r * nbg;
  const int b0 = bg * bper, b1 = min(B, b0 + bper);
  const int s0 = rseg_ptr[r], s1 = rseg_ptr[r + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = warp * NPW;
  float acc[NPW][F];
#pragma unroll
  for (int k = 0; k < NPW; ++k)
#pragma unroll
    for (int f = 0; f < F; ++f) acc[k][f] = 0.f;
  if (n0 < H) {
    for (int b = b0; b < b1; ++b) {
      for (int si = s0 + lane; si < s1; si += 32) {
        const int s = __ldg(rseg_list + si);
        const long long q = (long long)b * N + __ldg(seg_node + s);
        const int qt = (int)(q >> 7), rr = (int)(q & 127);
        const float* dcol = DT + (((size_t)qt * 4 + (rr >> 5)) * Ktot + col0 + n0) * 32 + (rr & 31);   // [tp][row quarter][col][32 rows]
        const float* urow = Ut + ((size_t)b * nseg + s) * F;
#pragma unroll 2
        for (int t = 0; t < T; ++t) {
          const float4 ua = __ldg(reinterpret_cast<const float4*>(urow + (size_t)t * B * nseg * F));
          const float4 ub = __ldg(reinterpret_cast<const float4*>(urow + (size_t)t * B * nseg * F) + 1);
          const float u[F] = {ua.x, ua.y, ua.z, ua.w, ub.x, ub.y, ub.z, ub.w};
          const float* dp = dcol + (size_t)t * nqt * 4 * Ktot * 32;
          float d[NPW];
#pragma unroll
          for (int k = 0; k < NPW; ++k) d[k] = __ldg(dp + (size_t)k * 32);
#pragma unroll
          for (int k = 0; k < NPW; ++k)
#pragma unroll
            for (int f = 0; f < F; ++f) acc[k][f] = fmaf(d[k], u[f], acc[k][f]);
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < NPW; ++k)
#pragma unroll
    for (int f = 0; f < F; ++f) {
      float v = acc[k][f];
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
      acc[k][f] = v;
    }
  if (lane == 0 && n0 < H) {
    float* o = part + ((size_t)c * H + n0) * F;
#pragma unroll
    for (int k = 0; k < NPW; ++k) {
      *reinterpret_cast<float4*>(o + k * F) = make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]);
      *reinterpret_cast<float4*>(o + k * F + 4) = make_float4(acc[k][4], acc[k][5], acc[k][6], acc[k][7]);
    }
  }
}
__global__ void k_m1_chunks_even(int R, int nbg, int32_t* __restrict__ chunk_ptr) {
  for (int r = threadIdx.x; r <= R; r += blockDim.x) chunk_ptr[r] = r * nbg;
}
// dM1[r][n][f] = sum of the region's chunk partials, in chunk order (zero for a region without segments)
__global__ void __launch_bounds__(256) k_m1_reduce(const float* __restrict__ part, const int32_t* __restrict__ chunk_ptr, int HF,
                                                   float* __restrict__ dM1) {
  const int r = blockIdx.x;
  const int c0 = chunk_ptr[r], c1 = chunk_ptr[r + 1];
  for (int i = threadIdx.x; i < HF; i += blockDim.x) {
    float s = 0.f;
    for (int c = c0; c < c1; ++c) s += part[(size_t)c * HF + i];
    dM1[(size_t)r * HF + i] = s;
  }
}

// ------------------------------------------------------------------------------------------
// shared split-K kernels
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_wgrad_tn(TNBatch batch, long long rows, int splits, long long chunk) {
  __shared__ __align__(16) float As[KT][TN];
  __shared__ __align__(16) float Bs[KT][TN];
  const int prob = blockIdx.z / splits, split = blockIdx.z - prob * splits;
  const TNProb p = batch.p[prob];
  const int m0 = blockIdx.y * TN, n0 = blockIdx.x * TN;
  if (m0 >= p.M || n0 >= p.N) return;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const long long r0 = split * chunk, r1 = min(rows, r0 + chunk);
  float acc[4][4];
  zero_acc(acc);
  for (long long rk = r0; rk < r1; rk += KT) {
    __syncthreads();
    for (int i = tid; i < KT * TN; i += 256) {
      const int kk = i / TN, c = i - kk * TN;
      const long long r = rk + kk;
      float va = 0.f, vb = 0.f;
      if (r < r1) {
        if (m0 + c < p.M) va = __ldg(p.A + r * p.lda + m0 + c);
        if (n0 + c < p.N) {
          vb = __ldg(p.B + r * p.ldb + n0 + c);
          if (p.relu_b) vb = fmaxf(vb, 0.f);
        }
      }
      As[kk][c] = va;
      Bs[kk][c] = vb;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < KT; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(av[i], b4.x, acc[i][0]);
        acc[i][1] = fmaf(av[i], b4.y, acc[i][1]);
        acc[i][2] = fmaf(av[i], b4.z, acc[i][2]);
        acc[i][3] = fmaf(av[i], b4.w, acc[i][3]);
      }
    }
  }
  float* o = p.part + (size_t)split * p.M * p.N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < p.N) o[(size_t)m * p.N + n] = acc[i][j];
    }
  }
}

int launch_wgrad_tn(const TNBatch& batch, long long rows, int splits, cudaStream_t st) {
  int maxM = 0, maxN = 0;
  for (int i = 0; i < batch.nprob; ++i) {
    maxM = max(maxM, batch.p[i].M);
    maxN = max(maxN, batch.p[i].N);
  }
  long long chunk = (rows + splits - 1) / splits;
  chunk = (chunk + KT - 1) / KT * KT;
  dim3 grid(cdiv(maxN, TN), cdiv(maxM, TN), batch.nprob * splits);
  k_wgrad_tn<<<grid, 256, 0, st>>>(batch, rows, splits, chunk);
  REGT_LAUNCHED("k_wgrad_tn", st);
  return 0;
}

__global__ void k_reduce_splits(const float* __restrict__ part, float* __restrict__ out, long long count, int splits,
                                int accumulate) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= count) return;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += part[(size_t)sp * count + i];
  out[i] = accumulate ? out[i] + s : s;
}
int launch_reduce_splits(const float* part, float* out, long long count, int splits, int accumulate, cudaStream_t st) {
  if (!out || count == 0) return 0;
  k_reduce_splits<<<cdiv(count, 256), 256, 0, st>>>(part, out, count, splits, accumulate);
  REGT_LAUNCHED("k_reduce_splits", st);
  return 0;
}

// part[split][c] = sum over the rows of the split of A[r][c].  256 threads = RS row lanes x CW column lanes
// (CW = power of two >= min(C, 128)): independent loads in flight, then a fixed-order sum over the row lanes.
__global__ void __launch_bounds__(256) k_colsum(const float* __restrict__ A, int lda, int C, long long rows,
                                                long long chunk, float* __restrict__ part, int CW) {
  __shared__ float red[256];
  const int RS = 256 / CW;
  const int cl = threadIdx.x % CW, rl = threadIdx.x / CW;
  const int c = blockIdx.x * CW + cl;
  const long long r0 = blockIdx.y * chunk, r1 = min(rows, r0 + chunk);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (c < C) {
    long long r = r0 + rl;
    for (; r + 3ll * RS < r1; r += 4ll * RS) {
      s0 += __ldg(A + r * lda + c);
      s1 += __ldg(A + (r + RS) * lda + c);
      s2 += __ldg(A + (r + 2ll * RS) * lda + c);
      s3 += __ldg(A + (r + 3ll * RS) * lda + c);
    }
    for (; r < r1; r += RS) s0 += __ldg(A + r * lda + c);
  }
  red[threadIdx.x] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (rl == 0 && c < C) {
    float s = 0.f;
    for (int i = 0; i < RS; ++i) s += red[i * CW + cl];
    part[(size_t)blockIdx.y * C + c] = s;
  }
}
int launch_colsum(const float* A, int lda, int C, long long rows, int splits, float* part, cudaStream_t st) {
  long long chunk = (rows + splits - 1) / splits;
  int CW = 1;
  while (CW < C && CW < 128) CW <<= 1;
  k_colsum<<<dim3(cdiv(C, CW), splits), 256, 0, st>>>(A, lda, C, rows, chunk, part, CW);
  REGT_LAUNCHED("k_colsum", st);
  return 0;
}

// ------------------------------------------------------------------------------------------
// host-side orchestration of the fp32 path
// ------------------------------------------------------------------------------------------

static CellK make_cellk(const regt_args* a, const Layout& L) {
  CellK k{};
  k.rows = a->B * a->N * a->T;
  k.N = a->N; k.xN = a->x_rows > 0 ? a->x_rows : a->N; k.T = a->T; k.H = a->H; k.nseg = a->plan.nseg; k.mode = a->mode;
  k.x = x_wide(a, L); k.S = L.S; k.U = L.U; k.h_ext = a->h_ext;
  k.seg_ptr = a->plan.seg_ptr; k.seg_reg = a->plan.seg_reg;
  k.M0t = L.M0t; k.M1t = L.M1t; k.c0 = L.c0; k.Wzr = L.Wzr; k.Wc = L.Wc; k.czr = L.czr; k.cc = L.cc; k.probs = L.probs;
  k.h = L.h; k.Z = L.Z; k.Rg = L.Rg; k.Hc = L.Hc; k.hR = L.hR; k.Hn = L.Hn;
  k.G = L.G; k.D = L.D; k.d_h_ext = a->d_h_ext;
  for (int g = 0; g < 3; ++g) k.lin_w[g] = a->p.lin_w[g];
  return k;
}

template <int TM>
static int run_fwd(const CellK& k, cudaStream_t st) {
  const size_t smem = ((size_t)2 * TM * (F + k.H + 1) + KT * TN) * sizeof(float);
  REGT_CUDA(cudaFuncSetAttribute(k_cell_fwd<TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_cell_fwd<TM><<<cdiv(k.rows, TM), TM * 4, smem, st>>>(k);
  REGT_LAUNCHED("k_cell_fwd", st);
  return 0;
}
template <int TM>
static int run_bwd(const CellK& k, cudaStream_t st) {
  const size_t smem = ((size_t)4 * TM * (k.H + 1) + 4 + KT * TN) * sizeof(float);
  REGT_CUDA(cudaFuncSetAttribute(k_cell_bwd<TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_cell_bwd<TM><<<cdiv(k.rows, TM), TM * 4, smem, st>>>(k);
  REGT_LAUNCHED("k_cell_bwd", st);
  return 0;
}

// dM1[r] = sum over the (node, region r) segments of dhp^T U; dhp = rows of `ldd` floats
static int launch_wgrad_m1_from(const regt_args* a, const Layout& L, const float* dhp, long long ldd, cudaStream_t st, int period_major,
                         long long BNp) {
  const int H = a->H, T = a->T, R = a->plan.R;
  const long long nsg = a->plan.nseg;
  const M1Strides sd = period_major ? M1Strides{ldd, BNp * ldd, nsg * F, F, 1, (long long)a->B * nsg * F}
                                    : M1Strides{(long long)T * ldd, ldd, nsg * F * T, (long long)F * T, T, 1};
  REGT_CHECK(H % 4 == 0 && ldd % 4 == 0 && ((uintptr_t)dhp % 16) == 0, "wgrad_m1: H and the row pitch must be multiples of 4 floats");
  const long long total = (long long)a->plan.nseg * a->B;
  const int per = (int)max(8ll, (total + M1_TARGET_CHUNKS - 1) / M1_TARGET_CHUNKS);
  const int max_chunks = (int)(total / per) + R + 1;
  REGT_CHECK((size_t)max_chunks * H * F <= L.part_floats, "wgrad_m1: partial buffer too small (%d chunks)", max_chunks);
  k_m1_chunks<<<1, 1024, 0, st>>>(a->plan.rseg_ptr, R, a->B, per, L.m1cp);
  REGT_LAUNCHED("k_m1_chunks", st);
  if (period_major) {
    const long long u_ts = (long long)a->B * nsg * F;
    if (T % 6 == 0)
      k_wgrad_m1_pm<6><<<dim3(max_chunks, cdiv(H, 128)), 128, 0, st>>>(dhp, ldd, BNp * ldd, L.U, u_ts, a->plan.rseg_ptr, a->plan.rseg_list,
                                                                     a->plan.seg_node, L.m1cp, a->B, a->N, T, H, R, a->plan.nseg, per, L.part);
    else
      k_wgrad_m1_pm<4><<<dim3(max_chunks, cdiv(H, 128)), 128, 0, st>>>(dhp, ldd, BNp * ldd, L.U, u_ts, a->plan.rseg_ptr, a->plan.rseg_list,
                                                                     a->plan.seg_node, L.m1cp, a->B, a->N, T, H, R, a->plan.nseg, per, L.part);
  } else if (T % 6 == 0)
    k_wgrad_m1<6><<<dim3(max_chunks, cdiv(H, 128)), 128, 0, st>>>(dhp, sd, L.U, a->plan.rseg_ptr, a->plan.rseg_list, a->plan.seg_node,
                                                                L.m1cp, a->B, a->N, T, H, R, a->plan.nseg, per, L.part);
  else
    k_wgrad_m1<4><<<dim3(max_chunks, cdiv(H, 128)), 128, 0, st>>>(dhp, sd, L.U, a->plan.rseg_ptr, a->plan.rseg_list, a->plan.seg_node,
                                                                L.m1cp, a->B, a->N, T, H, R, a->plan.nseg, per, L.part);
  REGT_LAUNCHED("k_wgrad_m1", st);
  k_m1_reduce<<<R, 256, 0, st>>>(L.part, L.m1cp, H * F, L.dM1);
  REGT_LAUNCHED("k_m1_reduce", st);
  return 0;
}
// dM1 from the transposed gate-gradient tiles of the fused backward: DT [T * nqt][Ktot = 4H][128], dhp = columns [3H, 4H)
int launch_wgrad_m1_kt(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, T = a->T, R = a->plan.R, B = a->B;
  REGT_CHECK(H % 16 == 0 && H <= 128, "wgrad_m1_kt: hidden %d not supported", H);
  const long long BN = (long long)B * a->N;
  const int nqt = (int)((BN + 127) / 128);
  int nbg = min(B, max(1, 2048 / max(R, 1)));
  const int bper = (B + nbg - 1) / nbg;
  nbg = (B + bper - 1) / bper;
  REGT_CHECK((size_t)R * nbg * H * F <= L.part_floats, "wgrad_m1_kt: partial buffer too small");
  k_m1_chunks_even<<<1, 256, 0, st>>>(R, nbg, L.m1cp);
  REGT_LAUNCHED("k_m1_chunks", st);
  if (H == 128)
    k_wgrad_m1_kt<8><<<R * nbg, 512, 0, st>>>(L.D, 4 * H, 3 * H, L.U, a->plan.rseg_ptr, a->plan.rseg_list, a->plan.seg_node, B, a->N, T,
                                              nqt, a->plan.nseg, nbg, bper, H, L.part);
  else
    k_wgrad_m1_kt<4><<<R * nbg, 512, 0, st>>>(L.D, 4 * H, 3 * H, L.U, a->plan.rseg_ptr, a->plan.rseg_list, a->plan.seg_node, B, a->N, T,
                                              nqt, a->plan.nseg, nbg, bper, H, L.part);
  REGT_LAUNCHED("k_wgrad_m1_kt", st);
  k_m1_reduce<<<R, 256, 0, st>>>(L.part, L.m1cp, H * F, L.dM1);
  REGT_LAUNCHED("k_m1_reduce", st);
  return 0;
}
int launch_wgrad_m1(const regt_args* a, const Layout& L, cudaStream_t st) {
  return launch_wgrad_m1_from(a, L, L.D + 3 * (size_t)a->H, 4ll * a->H, st, 0, 0);
}

// F-wide weight gradients (dP_g = D_g^T S, dM0 = D_3^T X, biases = column sums, dM1 per region)
static int launch_fwide_wgrads(const regt_args* a, const Layout& L, int splits, cudaStream_t st) {
  const int H = a->H, T = a->T, R = a->plan.R;
  const long long rows = (long long)a->B * a->N * T;
  float* part = L.part;
  const int ncol = (a->mode == REGT_MODE_TGCN) ? 3 * H : 4 * H;
  long long chunk = (rows + splits - 1) / splits;
  k_wgrad_skinny<<<dim3(cdiv(ncol, 128), splits), 128, 0, st>>>(L.D, L.S, x_wide(a, L), a->N, a->x_rows > 0 ? a->x_rows : a->N, H, T, rows, ncol, chunk, part);
  REGT_LAUNCHED("k_wgrad_skinny", st);
  k_skinny_reduce<<<cdiv((long long)ncol * (F + 1), 256), 256, 0, st>>>(part, splits, H, ncol, L.dP, L.dcg, L.dM0, L.dc0);
  REGT_LAUNCHED("k_skinny_reduce", st);
  if (a->mode != REGT_MODE_TGCN && launch_wgrad_m1(a, L, st)) return -1;
  return 0;
}

int cell_forward_fp32(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, T = a->T;
  const long long BN = (long long)a->B * a->N;
  const int xN = a->x_rows > 0 ? a->x_rows : a->N;
  if (launch_prep(a, L, st)) return -1;
  if (launch_widen_x(a, L, st)) return -1;
  // F-wide SpMM: S = A_hat X on rows of F*T floats; U per (node, region) segment
  if (launch_spmm_rows(a->plan.g_rowptr, a->plan.g_col, a->plan.g_val, x_wide(a, L), L.S, a->B, a->N, xN, F * T, st)) return -1;
  if (a->mode != REGT_MODE_TGCN && a->plan.nseg > 0) {
    if (launch_spmm_rows(a->plan.seg_eptr, a->plan.c_col, a->plan.c_val, x_wide(a, L), L.U, a->B, a->plan.nseg, xN, F * T, st))
      return -1;
  }
  CellK k = make_cellk(a, L);
  const size_t smem64 = ((size_t)2 * 64 * (F + H + 1) + KT * TN) * sizeof(float);
  int rc = (smem64 <= 200 * 1024) ? run_fwd<64>(k, st) : run_fwd<32>(k, st);
  if (rc) return rc;
  k_attn_accum<<<cdiv(BN * (H / 4), 256), 256, 0, st>>>(L.Hn, L.probs, T, H, BN, a->out_hidden);
  REGT_LAUNCHED("k_attn_accum", st);
  return 0;
}

int cell_backward_fp32(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, T = a->T, R = a->plan.R;
  const long long BN = (long long)a->B * a->N, rows = BN * T;
  CellK k = make_cellk(a, L);
  const size_t smem64 = ((size_t)4 * 64 * (H + 1) + 4 + KT * TN) * sizeof(float);
  int rc = (smem64 <= 200 * 1024) ? run_bwd<64>(k, st) : run_bwd<32>(k, st);
  if (rc) return rc;
  float* part = L.part;
  // attention gradient
  const int nblk = 128;
  k_dprobs<<<nblk, 256, 0, st>>>(L.G, L.Hn, T, H, BN, part);
  REGT_LAUNCHED("k_dprobs", st);
  if (launch_reduce_splits(part, L.dprobs, T, nblk, 0, st)) return -1;
  // H x H weight gradients: dB_z = Dz^T h, dB_r = Dr^T h, dB_h = Dh^T (h*R)
  const int splits = (int)max(1ll, min((long long)WGRAD_SPLITS, rows / 256));
  TNBatch tb{};
  tb.nprob = 3;
  for (int g = 0; g < 3; ++g) {
    tb.p[g].A = L.D + (size_t)g * H;
    tb.p[g].lda = 4 * H;
    tb.p[g].B = (g == 2) ? L.hR : L.h;
    tb.p[g].ldb = H;
    tb.p[g].M = H;
    tb.p[g].N = H;
    tb.p[g].relu_b = 0;
    tb.p[g].part = part + (size_t)g * splits * H * H;
  }
  if (launch_wgrad_tn(tb, rows, splits, st)) return -1;
  for (int g = 0; g < 3; ++g)
    if (launch_reduce_splits(tb.p[g].part, L.dB + (size_t)g * H * H, (long long)H * H, splits, 0, st)) return -1;
  if (launch_fwide_wgrads(a, L, splits, st)) return -1;
  return launch_chain(a, L, st);
}

}  // namespace regt
