// Decoder head in fp32-equivalent tensor-core arithmetic (precision tf32x3): the two 128-wide GEMMs of
//   out = linear2(relu(linear1(relu(out_hidden))))      models/RegionalTemporalGCN.py:35-38, models/TemporalGCN.py:28-31
// and of its backward run on the TMA-fed 3xTF32 GEMM of gemm_tma.cu (A through TMEM) instead of the FFMA tiles of head.cu
// (config 5: k_head_fwd + k_head_bwd + k_wgrad_tn = 33 ms of a 320 ms step, FFMA-bound), with three light row kernels around:
//   forward   rh = relu(hid)                                k_hf_relu
//             a1pre = rh . W1^T                             gemm_nt (tensor cores)
//             a1 = relu(a1pre + b1); out = a1 . W2^T + b2;  k_hf_mid   (warp per row; O <= 16 outputs through shuffles)
//             loss = sum (out - y)^2 / (N O), d_out         (run.py:180)
//   backward  d_a1 = (d_out . W2) * (a1 > 0); [d_out | 1] plane     k_hf_da1   (warp per row)
//             Gpre = d_a1 . W1                              gemm_nt (tensor cores)
//             G = Gpre * (hid > 0) + d_hidden               k_hf_gmask (row major or the tile layout the fused cell reads)
//             dW1, db1 = d_a1^T [relu(hid) | 1]             gemm_tn (tensor cores, as before)
//             dW2, (colsum a1) = a1^T [d_out | 1]           gemm_tn, feature-plane operand only
//             db2 = colsum d_out                            k_colsum
#include "common.cuh"

namespace regt {

namespace {
__global__ void __launch_bounds__(256) k_hf_relu(const float4* __restrict__ hid, float4* __restrict__ rh, long long n4) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 v = __ldg(hid + i);
  rh[i] = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
}

// warp per row; lane owns columns 4*lane .. 4*lane+3 of the 128-wide hidden layer
constexpr int HF_O = 16;     // output_dim handled by the shuffle reductions
__global__ void __launch_bounds__(256) k_hf_mid(float* __restrict__ a1, const float* __restrict__ b1, const float* __restrict__ w2,
                                                const float* __restrict__ b2, const float* __restrict__ y, long long BN, int O, float scale,
                                                float* __restrict__ out, float* __restrict__ d_out, float* __restrict__ loss_part) {
  __shared__ float red[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float w[HF_O][4];
#pragma unroll
  for (int o = 0; o < HF_O; ++o) {
    const float4 t = o < O ? __ldg(reinterpret_cast<const float4*>(w2 + (size_t)o * HEAD_HID) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    w[o][0] = t.x; w[o][1] = t.y; w[o][2] = t.z; w[o][3] = t.w;
  }
  const float4 bb = __ldg(reinterpret_cast<const float4*>(b1) + lane);
  float lsum = 0.f;
  // grid-stride over the rows (a bounded number of blocks: the loss partials are summed by one thread per output)
  for (long long q = blockIdx.x * 8ll + warp; q < BN; q += (long long)gridDim.x * 8) {
    const float4 p = reinterpret_cast<const float4*>(a1 + q * HEAD_HID)[lane];
    const float a[4] = {fmaxf(p.x + bb.x, 0.f), fmaxf(p.y + bb.y, 0.f), fmaxf(p.z + bb.z, 0.f), fmaxf(p.w + bb.w, 0.f)};
    reinterpret_cast<float4*>(a1 + q * HEAD_HID)[lane] = make_float4(a[0], a[1], a[2], a[3]);
    // 16 partial dot products per lane -> out[o] on lanes 2o, 2o+1 by a halving exchange: 8 + 4 + 2 + 1 + 1 = 16 shuffles per row
    // (a full butterfly per output was 80; the kernel is shuffle-bound).  Fixed order: deterministic.
    float s16[HF_O];
#pragma unroll
    for (int o = 0; o < HF_O; ++o) {
      float s = a[0] * w[o][0];
      s = fmaf(a[1], w[o][1], s); s = fmaf(a[2], w[o][2], s); s = fmaf(a[3], w[o][3], s);
      s16[o] = s;
    }
    float s8[8], s4[4], s2[2];
    {
      const bool up = lane & 16;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float keep = up ? s16[i + 8] : s16[i], send = up ? s16[i] : s16[i + 8];
        s8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
      }
    }
    {
      const bool up = lane & 8;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float keep = up ? s8[i + 4] : s8[i], send = up ? s8[i] : s8[i + 4];
        s4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
      }
    }
    {
      const bool up = lane & 4;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float keep = up ? s4[i + 2] : s4[i], send = up ? s4[i] : s4[i + 2];
        s2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
    }
    float mine;
    {
      const bool up = lane & 2;
      const float keep = up ? s2[1] : s2[0], send = up ? s2[0] : s2[1];
      mine = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    mine += __shfl_xor_sync(0xffffffffu, mine, 1);
    const int o = lane >> 1;     // lanes 2o and 2o+1 hold out[o] (bits 4..1 of the lane picked the halves)
    if ((lane & 1) == 0 && o < O) {
      const float v = mine + __ldg(b2 + o);
      out[q * O + o] = v;
      if (y) {
        const float diff = v - __ldg(y + q * O + o);
        lsum = fmaf(diff, diff, lsum);
        d_out[q * O + o] = 2.0f * diff * scale;
      }
    }
  }
  if (y) {   // fixed-order sums: lanes of a warp, then the eight warps
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, d);
    if (lane == 0) red[warp] = lsum;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s += red[i];
      loss_part[blockIdx.x] = s * scale;
    }
  }
}

// d_a1 = (d_out . W2) * (a1 > 0);  dO32[q] = [d_out(O) | 0.. | 1 at column 16 | 0..]
__global__ void __launch_bounds__(256) k_hf_da1(const float* __restrict__ a1, const float* __restrict__ w2, const float* __restrict__ d_out,
                                                long long BN, int O, float* __restrict__ d_a1, float* __restrict__ dO32) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long q = blockIdx.x * 8ll + warp;
  if (q >= BN) return;
  const float dv = lane < O ? __ldg(d_out + q * O + lane) : 0.f;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int o = 0; o < HF_O; ++o) {
    if (o < O) {
      const float d = __shfl_sync(0xffffffffu, dv, o);
      const float4 t = __ldg(reinterpret_cast<const float4*>(w2 + (size_t)o * HEAD_HID) + lane);
      acc[0] = fmaf(d, t.x, acc[0]); acc[1] = fmaf(d, t.y, acc[1]); acc[2] = fmaf(d, t.z, acc[2]); acc[3] = fmaf(d, t.w, acc[3]);
    }
  }
  const float4 a = __ldg(reinterpret_cast<const float4*>(a1 + q * HEAD_HID) + lane);
  reinterpret_cast<float4*>(d_a1 + q * HEAD_HID)[lane] =
      make_float4(a.x > 0.f ? acc[0] : 0.f, a.y > 0.f ? acc[1] : 0.f, a.z > 0.f ? acc[2] : 0.f, a.w > 0.f ? acc[3] : 0.f);
  dO32[q * 32 + lane] = lane < O ? dv : (lane == 16 ? 1.0f : 0.f);
}

// G = Gpre * (hid > 0) + d_hidden, four columns per thread
__global__ void __launch_bounds__(256) k_hf_gmask(const float4* __restrict__ gpre, const float4* __restrict__ hid, const float4* __restrict__ dh,
                                                  long long BN, int H, int tiled, float* __restrict__ G) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int h4 = H >> 2;
  if (i >= BN * h4) return;
  const long long q = i / h4;
  const int n = (int)(i - q * h4) * 4;
  const float4 g = __ldg(gpre + i), h = __ldg(hid + i);
  float4 v = make_float4(h.x > 0.f ? g.x : 0.f, h.y > 0.f ? g.y : 0.f, h.z > 0.f ? g.z : 0.f, h.w > 0.f ? g.w : 0.f);
  if (dh) {
    const float4 d = __ldg(dh + i);
    v.x += d.x; v.y += d.y; v.z += d.z; v.w += d.w;
  }
  *reinterpret_cast<float4*>(G + g_off(q, n, H, tiled)) = v;
}
// W1t[k][m] = w1[m][k]   (K-major operand of the data-gradient GEMM)
__global__ void k_hf_w1t(const float* __restrict__ w1, int H, float* __restrict__ W1t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * HEAD_HID) return;
  const int k = i / HEAD_HID, m = i % HEAD_HID;
  W1t[i] = w1[(size_t)m * H + k];
}
// dW2[o][n] (+)= sum over splits of C2[z][n][o] ;  C2 = partials of a1^T [d_out | 1]
__global__ void k_hf_dw2(const float* __restrict__ C2, int splits, int O, int acc, float* __restrict__ dW2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= O * HEAD_HID || !dW2) return;
  const int o = i / HEAD_HID, n = i % HEAD_HID;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += C2[((size_t)z * HEAD_HID + n) * 32 + o];
  dW2[i] = acc ? dW2[i] + s : s;
}
}  // namespace

bool head_f_fits(int O) { return O <= HF_O; }

int head_forward_f(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, O = a->O;
  const long long BN = (long long)a->B * a->N;
  const int Nl = a->loss_nodes > 0 ? a->loss_nodes : a->N;
  k_hf_relu<<<cdiv(BN * H / 4, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(a->out_hidden), reinterpret_cast<float4*>(L.hf_rh), BN * H / 4);
  REGT_LAUNCHED("k_hf_relu", st);
  if (launch_gemm_nt_tma(L.hf_rh, H, a->p.head_w1, H, L.a1, HEAD_HID, BN, HEAD_HID, H, L.hf_split, st)) return -1;
  const int nblk = (int)min((long long)cdiv(BN, 8), 1184ll);      // 8 blocks per SM, grid-stride
  REGT_CHECK(!a->y || (a->loss && a->d_out), "head_forward: y given but loss/d_out is NULL");
  REGT_CHECK(!a->y || (size_t)nblk <= L.hf_loss_floats, "head_forward: loss partial buffer too small");
  k_hf_mid<<<nblk, 256, 0, st>>>(L.a1, a->p.head_b1, a->p.head_w2, a->p.head_b2, a->y, BN, O, 1.0f / ((float)Nl * (float)O), a->out,
                                 a->d_out, L.hf_loss);
  REGT_LAUNCHED("k_hf_mid", st);
  if (a->y) return launch_reduce_splits(L.hf_loss, a->loss, 1, nblk, 0, st);
  return 0;
}

int head_backward_f(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, O = a->O;
  const long long BN = (long long)a->B * a->N;
  k_hf_da1<<<cdiv(BN, 8), 256, 0, st>>>(L.a1, a->p.head_w2, a->d_out, BN, O, L.d_a1, L.hf_do32);
  REGT_LAUNCHED("k_hf_da1", st);
  float* W1t = L.part + L.part_floats - (size_t)H * HEAD_HID;     // [H][128], tail of the split-K scratch
  k_hf_w1t<<<cdiv((long long)H * HEAD_HID, 256), 256, 0, st>>>(a->p.head_w1, H, W1t);
  REGT_LAUNCHED("k_hf_w1t", st);
  // Gpre[q][k] = sum_n d_a1[q][n] W1[n][k]
  if (launch_gemm_nt_tma(L.d_a1, HEAD_HID, W1t, HEAD_HID, L.hf_rh, H, BN, H, HEAD_HID, L.hf_split, st)) return -1;
  k_hf_gmask<<<cdiv(BN * (H / 4), 256), 256, 0, st>>>(reinterpret_cast<const float4*>(L.hf_rh), reinterpret_cast<const float4*>(a->out_hidden),
                                                      reinterpret_cast<const float4*>(a->d_hidden), BN, H, L.route.g_tiled, L.G);
  REGT_LAUNCHED("k_hf_gmask", st);
  // weight gradients: row contractions on the tensor cores, split over the rows so that the grid fills the SMs
  float* part = L.part;
  if (launch_head_dw1_tf32x3(a, L, L.hf_do32, st)) return -1;   // [d_out | 1]: column 16 is the ones column
  const int s2 = (int)max(1ll, min(148ll, BN / 256));
  float* p3 = part;                                    // [s2][128][32]   a1^T [d_out | 1]
  if (launch_gemm_tn(L.a1, HEAD_HID, nullptr, 0, nullptr, BN, HEAD_HID, 0, s2, st, L.hf_do32, 32, p3, 0, 0)) return -1;
  k_hf_dw2<<<cdiv(O * HEAD_HID, 256), 256, 0, st>>>(p3, s2, O, a->accumulate, a->g.head_w2);
  REGT_LAUNCHED("k_hf_dw2", st);
  const int s3 = (int)max(1ll, min(128ll, BN / 128));
  if (launch_colsum(a->d_out, O, O, BN, s3, part, st)) return -1;
  return launch_reduce_splits(part, a->g.head_b2, O, s3, a->accumulate, st);
}

}  // namespace regt
