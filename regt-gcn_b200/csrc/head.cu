// Decoder head of RegionalTemporalGCN / TemporalGCN and the call-site loss:
//   out = linear2(relu(linear1(relu(out_hidden))))      models/RegionalTemporalGCN.py:35-38
//   loss = sum_b mean_{n,o} (out - y)^2                 run.py:180 (one backward per snapshot)
//          (or the MAE, or either over the valid targets only: LossX, common.cuh)
// plus their autograd (run.py:190).  One row per (b, n); tiny next to the cell.
#include "gemm_simt.cuh"

namespace regt {

constexpr int TMH = 64;

struct HeadK {
  long long BN;
  int N, H, O;   // N = node count of the loss mean (regt_args.loss_nodes or N)
  const float *hid, *y, *W1t, *W2t, *b1, *b2;  // W1t [H][128], W2t [128][O]
  const float *w1, *w2;                        // natural layouts for the data gradients
  const float* d_hidden;
  float *a1, *out, *d_out, *loss_part, *d_a1, *G;
  const float* hid_part;  // tensor-core cell: [ntc][nqt][H/4][128][4] partial attention sums (NULL: hid is final)
  int ntc, nqt;
  float* hid_out;         // where the summed out_hidden goes when hid_part is used
  int g_tiled;            // 1: G is written as [qt][H/4][128][4] tiles (tensor-core backward), 0: row-major
  LossX lx;               // loss kind and mask of the LX instantiations
};

__global__ void k_head_transpose(const float* __restrict__ w1, const float* __restrict__ w2, int H, int O,
                                 float* __restrict__ W1t, float* __restrict__ W2t) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < H * HEAD_HID) {
    int k = i / HEAD_HID, m = i % HEAD_HID;  // W1t[k][m] = w1[m][k]
    W1t[i] = w1[(size_t)m * H + k];
  } else if (i < H * HEAD_HID + HEAD_HID * O) {
    int j = i - H * HEAD_HID;
    int m = j / O, o = j % O;  // W2t[m][o] = w2[o][m]
    W2t[j] = w2[(size_t)o * HEAD_HID + m];
  }
}

template <bool LX>
__global__ void __launch_bounds__(TMH * 4) k_head_fwd(HeadK a) {
  constexpr int NT = TMH * 4;
  extern __shared__ __align__(16) float smem[];
  const int H = a.H, O = a.O, lda = H + 1, ld1 = HEAD_HID + 1;
  float* A0 = smem;                 // relu(hid) [TMH][H+1]
  float* A1 = A0 + TMH * lda;       // a1 [TMH][129]
  float* Ws = A1 + TMH * ld1;       // offsets are multiples of 64 floats
  __shared__ float red[32];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const long long q0 = (long long)blockIdx.x * TMH;
  for (int idx = tid; idx < TMH * H; idx += NT) {
    const int rl = idx / H, j = idx - rl * H;
    const long long q = q0 + rl;
    A0[rl * lda + j] = q < a.BN ? fmaxf(a.hid[q * H + j], 0.f) : 0.f;
  }
  for (int n0 = 0; n0 < HEAD_HID; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(A0, lda, H, a.W1t, HEAD_HID, n0, HEAD_HID, Ws, acc, ty, tx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rl = ty * 4 + i;
      const long long q = q0 + rl;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        const float v = fmaxf(acc[i][j] + __ldg(a.b1 + n), 0.f);
        A1[rl * ld1 + n] = v;
        if (q < a.BN) a.a1[q * HEAD_HID + n] = v;
      }
    }
  }
  float lsum = 0.f, lsc = 0.f;
  const float scale = 1.0f / ((float)a.N * (float)O);
  for (int n0 = 0; n0 < O; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(A1, ld1, HEAD_HID, a.W2t, O, n0, O, Ws, acc, ty, tx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long q = q0 + ty * 4 + i;
      if (q >= a.BN) continue;
      float inv = scale;
      if constexpr (LX) inv = lossx_inv(a.lx, q, scale);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n >= O) continue;
        const float v = acc[i][j] + __ldg(a.b2 + n);
        a.out[q * O + n] = v;
        if (a.y) {
          if constexpr (LX) {
            a.d_out[q * O + n] = lossx_elem(a.lx, v, __ldg(a.y + q * O + n), inv, scale, lsum, lsc);
          } else {
            const float diff = v - __ldg(a.y + q * O + n);
            lsum = fmaf(diff, diff, lsum);
            a.d_out[q * O + n] = 2.0f * diff * scale;
          }
        }
      }
    }
  }
  if (a.y) {
    lsum = block_sum(lsum, red);
    if constexpr (LX) {
      lsc = block_sum(lsc, red);
      if (tid == 0) a.loss_part[blockIdx.x] = lsum * scale + lsc;
    } else {
      if (tid == 0) a.loss_part[blockIdx.x] = lsum * scale;
    }
  }
}

__global__ void __launch_bounds__(TMH * 4) k_head_bwd(HeadK a) {
  constexpr int NT = TMH * 4;
  extern __shared__ __align__(16) float smem[];
  const int H = a.H, O = a.O, ldo = O + 1, ld1 = HEAD_HID + 1;
  float* Do = smem;                 // d_out [TMH][O+1]
  float* D1 = Do + TMH * ldo;       // d_a1 [TMH][129]
  float* Ws = D1 + TMH * ld1;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const long long q0 = (long long)blockIdx.x * TMH;
  for (int idx = tid; idx < TMH * O; idx += NT) {
    const int rl = idx / O, j = idx - rl * O;
    const long long q = q0 + rl;
    Do[rl * ldo + j] = q < a.BN ? a.d_out[q * O + j] : 0.f;
  }
  // d_a1 = (d_out . W2) * (a1 > 0)
  for (int n0 = 0; n0 < HEAD_HID; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(Do, ldo, O, a.w2, HEAD_HID, n0, HEAD_HID, Ws, acc, ty, tx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rl = ty * 4 + i;
      const long long q = q0 + rl;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        float v = 0.f;
        if (q < a.BN) {
          v = a.a1[q * HEAD_HID + n] > 0.f ? acc[i][j] : 0.f;
          a.d_a1[q * HEAD_HID + n] = v;
        }
        D1[rl * ld1 + n] = v;
      }
    }
  }
  // G = (d_a1 . W1) * (hid > 0) + d_hidden
  for (int n0 = 0; n0 < H; n0 += TN) {
    float acc[4][4];
    zero_acc(acc);
    tile_gemm<NT>(D1, ld1, HEAD_HID, a.w1, H, n0, H, Ws, acc, ty, tx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long q = q0 + ty * 4 + i;
      if (q >= a.BN) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n >= H) continue;
        float v = a.hid[q * H + n] > 0.f ? acc[i][j] : 0.f;
        if (a.d_hidden) v += a.d_hidden[q * H + n];
        a.G[g_off(q, n, H, a.g_tiled)] = v;
      }
    }
  }
}

// gradient flowing only through out_hidden (no head gradient): G = d_hidden or 0
__global__ void k_copy_or_zero(const float* __restrict__ src, float* __restrict__ dst, long long n, int H, int tiled) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) dst[g_off(i / H, (int)(i % H), H, tiled)] = src ? src[i] : 0.f;
}

// ------------------------------------------------------------------------------------------
// fused training head (fuse_head): forward + loss + data gradients + weight-gradient partials in
// ONE persistent kernel; weights stay in shared memory, dW1 accumulates in registers.
// ------------------------------------------------------------------------------------------
constexpr int HP_MAX_CTAS = 148;
// multiple of 4 floats: the tensor-core head writes its dW1 partial with 16-byte stores
__host__ __device__ inline int head_part_stride(int H, int O) { return (HEAD_HID * H + O * HEAD_HID + HEAD_HID + O + 4 + 3) & ~3; }

template <int H, bool LX>
__global__ void __launch_bounds__(256, 1) k_head_fused(HeadK a, float* __restrict__ hpart, int ntiles) {
  constexpr int HJ = H / 16;             // dW1 columns per thread
  constexpr int LDA = H + 4, LD1 = HEAD_HID + 4;
  extern __shared__ __align__(16) float smem[];
  const int O = a.O, OP = (O + 3) & ~3, LDO = OP + 4;
  float* W1t = smem;                      // [H][128]      linear1.weight^T
  float* W1n = W1t + H * HEAD_HID;        // [128][H]      linear1.weight
  float* W2t = W1n + HEAD_HID * H;        // [128][OP]     linear2.weight^T (zero padded)
  float* W2n = W2t + HEAD_HID * OP;       // [O][128]      linear2.weight
  float* A0 = W2n + O * HEAD_HID;         // [64][LDA]     relu(hid)
  float* A1 = A0 + TMH * LDA;             // [64][LD1]     a1
  float* D1 = A1 + TMH * LD1;             // [64][LD1]     d a1
  float* Do = D1 + TMH * LD1;             // [64][LDO]     d out
  float* W2acc = Do + TMH * LDO;          // [O][128]      dW2 accumulator
  __shared__ float red[32];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  for (int i = tid; i < HEAD_HID * H; i += 256) {
    const int m = i / H, k = i % H;
    const float v = __ldg(a.w1 + i);
    W1n[i] = v;
    W1t[k * HEAD_HID + m] = v;
  }
  for (int i = tid; i < HEAD_HID * OP; i += 256) {
    const int m = i / OP, o = i % OP;
    W2t[i] = o < O ? __ldg(a.w2 + (size_t)o * HEAD_HID + m) : 0.f;
  }
  for (int i = tid; i < O * HEAD_HID; i += 256) {
    W2n[i] = __ldg(a.w2 + i);
    W2acc[i] = 0.f;
  }
  float dw1[8][HJ];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < HJ; ++j) dw1[i][j] = 0.f;
  float dbias = 0.f, lsum = 0.f, lsc = 0.f;
  const float scale = 1.0f / ((float)a.N * (float)O);
  __syncthreads();

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long q0 = (long long)tile * TMH;
    // relu(hid) tile
    for (int i = tid; i < TMH * (H / 4); i += 256) {
      const int rl = i / (H / 4), c4 = i % (H / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q0 + rl < a.BN) {
        if (a.hid_part) {  // sum the per-chunk attention partials of the tensor-core cell (fixed order)
          for (int c = 0; c < a.ntc; ++c) {
            const long long q = q0 + rl;   // tiled partials [chunk][qt][H/4][128][4]
            const float4 p = __ldg(reinterpret_cast<const float4*>(a.hid_part) +
                                   (((size_t)c * a.nqt + (size_t)(q >> 7)) * (H / 4) + c4) * 128 + (q & 127));
            v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
          }
          reinterpret_cast<float4*>(a.hid_out + (q0 + rl) * H)[c4] = v;
        } else {
          v = __ldg(reinterpret_cast<const float4*>(a.hid + (q0 + rl) * H) + c4);
        }
      }
      float* d = A0 + rl * LDA + c4 * 4;
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;   // pre-activation kept: sign needed for d hid
    }
    __syncthreads();
    // a1 = relu(relu(hid) W1^T + b1)
    for (int n0 = 0; n0 < HEAD_HID; n0 += TN) {
      float acc[4][4];
      zero_acc(acc);
#pragma unroll 4
      for (int k = 0; k < H; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(W1t + k * HEAD_HID + n0 + tx * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float av = fmaxf(A0[(ty * 4 + i) * LDA + k], 0.f);
          acc[i][0] = fmaf(av, b.x, acc[i][0]); acc[i][1] = fmaf(av, b.y, acc[i][1]);
          acc[i][2] = fmaf(av, b.z, acc[i][2]); acc[i][3] = fmaf(av, b.w, acc[i][3]);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = n0 + tx * 4 + j;
          A1[(ty * 4 + i) * LD1 + n] = fmaxf(acc[i][j] + __ldg(a.b1 + n), 0.f);
        }
    }
    __syncthreads();
    // out = a1 W2^T + b2 ; loss ; d_out
    for (int n0 = 0; n0 < OP; n0 += TN) {
      float acc[4][4];
      zero_acc(acc);
      if (n0 + tx * 4 < OP) {
#pragma unroll 4
        for (int k = 0; k < HEAD_HID; ++k) {
          const float4 b = *reinterpret_cast<const float4*>(W2t + k * OP + n0 + tx * 4);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float av = A1[(ty * 4 + i) * LD1 + k];
            acc[i][0] = fmaf(av, b.x, acc[i][0]); acc[i][1] = fmaf(av, b.y, acc[i][1]);
            acc[i][2] = fmaf(av, b.z, acc[i][2]); acc[i][3] = fmaf(av, b.w, acc[i][3]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = ty * 4 + i;
        const long long q = q0 + rl;
        float inv = scale;
        if constexpr (LX) inv = q < a.BN ? lossx_inv(a.lx, q, scale) : scale;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = n0 + tx * 4 + j;
          if (n >= OP) continue;
          float dv = 0.f;
          if (n < O && q < a.BN) {
            const float v = acc[i][j] + __ldg(a.b2 + n);
            a.out[q * O + n] = v;
            if constexpr (LX) {
              dv = lossx_elem(a.lx, v, __ldg(a.y + q * O + n), inv, scale, lsum, lsc);
            } else {
              const float diff = v - __ldg(a.y + q * O + n);
              lsum = fmaf(diff, diff, lsum);
              dv = 2.0f * diff * scale;
            }
            a.d_out[q * O + n] = dv;
          }
          Do[rl * LDO + n] = dv;
        }
      }
    }
    __syncthreads();
    // d a1 = (d_out W2) * (a1 > 0)
    for (int n0 = 0; n0 < HEAD_HID; n0 += TN) {
      float acc[4][4];
      zero_acc(acc);
      for (int k = 0; k < O; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(W2n + k * HEAD_HID + n0 + tx * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float av = Do[(ty * 4 + i) * LDO + k];
          acc[i][0] = fmaf(av, b.x, acc[i][0]); acc[i][1] = fmaf(av, b.y, acc[i][1]);
          acc[i][2] = fmaf(av, b.z, acc[i][2]); acc[i][3] = fmaf(av, b.w, acc[i][3]);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int idx = (ty * 4 + i) * LD1 + n0 + tx * 4 + j;
          D1[idx] = A1[idx] > 0.f ? acc[i][j] : 0.f;
        }
    }
    __syncthreads();
    // G = (d a1 W1) * (hid > 0) (+ d_hidden)
    for (int n0 = 0; n0 < H; n0 += TN) {
      float acc[4][4];
      zero_acc(acc);
      if (n0 + tx * 4 >= H) continue;   // H < 64: the upper thread columns have no output
#pragma unroll 4
      for (int k = 0; k < HEAD_HID; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(W1n + k * H + n0 + tx * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float av = D1[(ty * 4 + i) * LD1 + k];
          acc[i][0] = fmaf(av, b.x, acc[i][0]); acc[i][1] = fmaf(av, b.y, acc[i][1]);
          acc[i][2] = fmaf(av, b.z, acc[i][2]); acc[i][3] = fmaf(av, b.w, acc[i][3]);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = ty * 4 + i;
        const long long q = q0 + rl;
        if (q >= a.BN) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = n0 + tx * 4 + j;
          v[j] = A0[rl * LDA + n] > 0.f ? acc[i][j] : 0.f;
          if (a.d_hidden) v[j] += a.d_hidden[q * H + n];
        }
        *reinterpret_cast<float4*>(a.G + g_off(q, n0 + tx * 4, H, a.g_tiled)) = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
    // weight gradients of this tile: dW1 += d a1^T relu(hid) (registers), dW2 += d_out^T a1 (smem), biases
    {
      const int m0 = (tid >> 4) * 8, j0 = (tid & 15) * HJ;
      for (int rl = 0; rl < TMH; ++rl) {
        float d[8], av[HJ];
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] = D1[rl * LD1 + m0 + i];
#pragma unroll
        for (int j = 0; j < HJ; ++j) av[j] = fmaxf(A0[rl * LDA + j0 + j], 0.f);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < HJ; ++j) dw1[i][j] = fmaf(d[i], av[j], dw1[i][j]);
      }
      for (int i = tid; i < O * HEAD_HID; i += 256) {
        const int o = i / HEAD_HID, m = i % HEAD_HID;
        float sacc = 0.f;
        for (int rl = 0; rl < TMH; ++rl) sacc = fmaf(Do[rl * LDO + o], A1[rl * LD1 + m], sacc);
        W2acc[i] += sacc;
      }
      if (tid < HEAD_HID) {
        for (int rl = 0; rl < TMH; ++rl) dbias += D1[rl * LD1 + tid];
      } else if (tid - HEAD_HID < O) {
        for (int rl = 0; rl < TMH; ++rl) dbias += Do[rl * LDO + tid - HEAD_HID];
      }
    }
    __syncthreads();
  }
  // per-CTA partials: dW1 | dW2 | db1 | db2 | loss
  float* hp = hpart + (size_t)blockIdx.x * head_part_stride(H, O);
  {
    const int m0 = (tid >> 4) * 8, j0 = (tid & 15) * HJ;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < HJ; ++j) hp[(m0 + i) * H + j0 + j] = dw1[i][j];
  }
  for (int i = tid; i < O * HEAD_HID; i += 256) hp[HEAD_HID * H + i] = W2acc[i];
  if (tid < HEAD_HID) hp[HEAD_HID * H + O * HEAD_HID + tid] = dbias;
  else if (tid - HEAD_HID < O) hp[HEAD_HID * H + O * HEAD_HID + HEAD_HID + tid - HEAD_HID] = dbias;
  lsum = block_sum(lsum, red);
  if constexpr (LX) {
    lsc = block_sum(lsc, red);
    if (tid == 0) hp[HEAD_HID * H + O * HEAD_HID + HEAD_HID + O] = lsum * scale + lsc;
  } else {
    if (tid == 0) hp[HEAD_HID * H + O * HEAD_HID + HEAD_HID + O] = lsum * scale;
  }
}

// sums the per-CTA partials into the head gradients; the slot after the gradients is the loss
__global__ void __launch_bounds__(256) k_head_grad_reduce(const float* __restrict__ hpart, int stride, int ncta, int H,
                                                          int O, int acc, float* __restrict__ gw1,
                                                          float* __restrict__ gw2, float* __restrict__ gb1,
                                                          float* __restrict__ gb2, float* __restrict__ loss) {
  __shared__ float red[8][32];
  const int i = blockIdx.x * 32 + threadIdx.x;
  const int n1 = HEAD_HID * H, n2 = O * HEAD_HID, ntot = n1 + n2 + HEAD_HID + O;
  const float s = sum_parts_32x8(hpart, stride, ncta, i, i <= ntot, red);
  if (threadIdx.y != 0 || i > ntot) return;
  if (i == ntot) {
    if (loss) *loss = s;
    return;
  }
  float* dst;
  int j = i;
  if (j < n1) dst = gw1;
  else if ((j -= n1) < n2) dst = gw2;
  else if ((j -= n2) < HEAD_HID) dst = gb1;
  else { j -= HEAD_HID; dst = gb2; }
  if (dst) dst[j] = acc ? dst[j] + s : s;
}

// k_head_fused keeps both weight layouts, the dW2 accumulator and four row tiles in shared memory
static size_t head_fused_smem(int H, int O) {
  const int OP = (O + 3) & ~3;
  return ((size_t)2 * HEAD_HID * H + HEAD_HID * OP + 2 * O * HEAD_HID + TMH * (H + 4) + 2 * TMH * (HEAD_HID + 4) +
          TMH * (OP + 4)) * sizeof(float);
}
// H = 64 fits up to O = 44 in the 227 KB a block may use (O = 45 would need 229 KB), H = 32 every O up to 64; wider
// heads run k_head_fwd / k_head_bwd
bool head_fused_fits(int H, int O) { return (H == 64 || H == 32) && O <= 64 && head_fused_smem(H, O) <= 227 * 1024; }
static int head_fused_grid(const regt_args* a) {
  const long long BN = (long long)a->B * a->N;
  return (int)min((long long)HP_MAX_CTAS, (BN + TMH - 1) / TMH);
}

int head_part_stride_host(int H, int O) { return head_part_stride(H, O); }
static HeadK make_headk(const regt_args* a, const Layout& L, float* W1t, float* W2t) {
  HeadK k{};
  k.BN = (long long)a->B * a->N;
  k.N = a->loss_nodes > 0 ? a->loss_nodes : a->N; k.H = a->H; k.O = a->O;
  k.hid = a->out_hidden; k.y = a->y; k.W1t = W1t; k.W2t = W2t; k.b1 = a->p.head_b1; k.b2 = a->p.head_b2;
  k.w1 = a->p.head_w1; k.w2 = a->p.head_w2; k.d_hidden = a->d_hidden;
  k.a1 = L.a1; k.out = a->out; k.d_out = a->d_out; k.loss_part = L.part; k.d_a1 = L.d_a1; k.G = L.G;
  k.hid_part = nullptr; k.ntc = 0; k.hid_out = a->out_hidden;
  k.g_tiled = L.route.g_tiled;
  k.lx = make_lossx(a, L);
  if (L.route.hid_partials) {  // the cell left per-chunk partials (see cell_tc.cu)
    k.hid_part = L.hid_part;
    k.ntc = tc_num_chunks(a);
    k.nqt = (int)((k.BN + 127) / 128);
  }
  return k;
}

// valid targets among rows [0, N) of y, counted as integers (exact in any order): block (chunk, b) writes the count of
// its slice of snapshot b to part[b][chunk]; k_loss_inv sums a snapshot's chunks and writes inv_c[b] = 1 / c_b (0 when
// c_b = 0), or takes c_b from the caller's counts
__global__ void __launch_bounds__(256) k_loss_count(const float* __restrict__ y, long long n, float null_v,
                                                    unsigned int* __restrict__ part) {
  __shared__ unsigned int red[8];
  const float* yb = y + (size_t)blockIdx.y * n;
  unsigned int k = 0;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float v = __ldg(yb + i);
    k += (v == v && v != null_v) ? 1u : 0u;
  }
  for (int d = 16; d > 0; d >>= 1) k += __shfl_xor_sync(0xffffffffu, k, d);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = k;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int s = 0;
    for (int w = 0; w < 8; ++w) s += red[w];
    part[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = s;
  }
}
__global__ void k_loss_inv(const unsigned int* __restrict__ part, int nchunks, const float* __restrict__ given, int B,
                           float* __restrict__ inv_c) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float c;
  if (given) {
    c = given[b];
  } else {
    unsigned long long k = 0;
    for (int i = 0; i < nchunks; ++i) k += part[(size_t)b * nchunks + i];
    c = (float)k;
  }
  inv_c[b] = c > 0.f ? 1.0f / c : 0.f;
}

LossX make_lossx(const regt_args* a, const Layout& L) {
  LossX x{};
  x.mae = a->loss_kind == REGT_LOSS_MAE;
  x.masked = a->loss_masked != 0;
  x.null_v = a->loss_null;
  x.inv_c = a->loss_masked ? L.inv_c : nullptr;
  x.N = a->N;
  return x;
}

int head_forward(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, O = a->O;
  if (a->y && a->loss_masked) {
    const long long n = (long long)a->N * O;
    const int nchunks = (int)min((long long)LC_CHUNKS, (n + 2047) / 2048);
    unsigned int* part = L.lc_part;
    if (!a->loss_count) {
      k_loss_count<<<dim3(nchunks, a->B), 256, 0, st>>>(a->y, n, a->loss_null, part);
      REGT_LAUNCHED("k_loss_count", st);
    }
    k_loss_inv<<<cdiv(a->B, 128), 128, 0, st>>>(part, nchunks, a->loss_count, a->B, L.inv_c);
    REGT_LAUNCHED("k_loss_inv", st);
  }
  switch (L.route.head) {
    case HeadPath::Bf16: return head_forward_tc(a, L, st);
    case HeadPath::Tf32x3: return head_forward_f(a, L, st);   // the 128-wide GEMMs on the tensor cores (head_f.cu)
    case HeadPath::FusedFfma: {
      HeadK k = make_headk(a, L, nullptr, nullptr);
      const int grid = head_fused_grid(a), ntiles = cdiv(k.BN, TMH);
      const size_t smem = head_fused_smem(H, O);
      auto kern = H == 64 ? (loss_ext(a) ? k_head_fused<64, true> : k_head_fused<64, false>)
                          : (loss_ext(a) ? k_head_fused<32, true> : k_head_fused<32, false>);
      REGT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kern<<<grid, 256, smem, st>>>(k, L.hpart, ntiles);
      REGT_LAUNCHED("k_head_fused", st);
      return 0;   // loss and head gradients are finalised by k_head_grad_reduce in regt_head_backward
    }
    case HeadPath::Rows: break;
  }
  // transposed head weights live at the tail of the split-K scratch's first page
  float* W1t = L.part + L.part_floats - ((size_t)H * HEAD_HID + (size_t)HEAD_HID * O);
  float* W2t = W1t + (size_t)H * HEAD_HID;
  k_head_transpose<<<cdiv((long long)H * HEAD_HID + HEAD_HID * O, 256), 256, 0, st>>>(a->p.head_w1, a->p.head_w2, H, O,
                                                                                  W1t, W2t);
  REGT_LAUNCHED("k_head_transpose", st);
  HeadK k = make_headk(a, L, W1t, W2t);
  const int nblk = cdiv(k.BN, TMH);
  const size_t smem = ((size_t)TMH * (H + 1) + TMH * (HEAD_HID + 1) + KT * TN) * sizeof(float);
  auto kern = loss_ext(a) ? k_head_fwd<true> : k_head_fwd<false>;
  REGT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<nblk, TMH * 4, smem, st>>>(k);
  REGT_LAUNCHED("k_head_fwd", st);
  if (a->y) {
    REGT_CHECK(a->loss && a->d_out, "head_forward: y given but loss/d_out is NULL");
    if (launch_reduce_splits(L.part, a->loss, 1, nblk, 0, st)) return -1;
  }
  return 0;
}

// out[r] (+)= sum over splits of Cp2[s][r][col]   (one column of a [splits][rows][32] partial array)
__global__ void k_pick_col(const float* __restrict__ Cp2, int splits, int rows, int col, int acc, float* __restrict__ out) {
  const int r = threadIdx.x;
  if (r >= rows || !out) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += Cp2[((size_t)z * rows + r) * 32 + col];
  out[r] = acc ? out[r] + s : s;
}

// dW1 = d_a1^T relu(hid) and, in the same pass over d_a1, db1 on the tensor cores (TMA-fed 3xTF32 row contraction): db1 is
// column 16 of d_a1^T ones, where `ones` is a [>= BN][32] plane whose column 16 is all ones, split over the rows to fill the SMs
int launch_head_dw1_tf32x3(const regt_args* a, const Layout& L, const float* ones, cudaStream_t st) {
  const int H = a->H;
  const long long BN = (long long)a->B * a->N;
  const int s1 = (int)max(1ll, min((long long)cdiv(148, cdiv(H, 128)), BN / 256));
  float* p1 = L.part;                                  // [s1][128][H]    d_a1^T relu(hid)
  float* p2 = L.part + (size_t)s1 * HEAD_HID * H;      // [s1][128][32]   d_a1^T ones  -> column 16 = db1
  if (launch_gemm_tn(L.d_a1, HEAD_HID, a->out_hidden, H, p1, BN, HEAD_HID, H, s1, st, ones, 32, p2, 0, 1)) return -1;
  if (launch_reduce_splits(p1, a->g.head_w1, (long long)HEAD_HID * H, s1, a->accumulate, st)) return -1;
  k_pick_col<<<1, HEAD_HID, 0, st>>>(p2, s1, HEAD_HID, 16, a->accumulate, a->g.head_b1);
  REGT_LAUNCHED("k_pick_col", st);
  return 0;
}

int launch_head_grad_reduce(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, O = a->O;
  const int stride = head_part_stride(H, O), n = HEAD_HID * H + O * HEAD_HID + HEAD_HID + O;
  const int ncta = L.route.head == HeadPath::Bf16 ? head_tc_grid(a) : head_fused_grid(a);
  k_head_grad_reduce<<<cdiv(n + 1, 32), dim3(32, 8), 0, st>>>(L.hpart, stride, ncta, H, O, a->accumulate, a->g.head_w1,
                                                            a->g.head_w2, a->g.head_b1, a->g.head_b2, a->loss);
  REGT_LAUNCHED("k_head_grad_reduce", st);
  return 0;
}

int head_backward(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, O = a->O;
  const long long BN = (long long)a->B * a->N;
  // fused heads: everything but the cross-CTA sum already happened in head_forward; the bf16 step runs that sum beside
  // the cell backward (launch_head_grad_reduce from cell_backward_tc)
  if (L.route.head == HeadPath::Bf16) return 0;
  if (L.route.head == HeadPath::FusedFfma) return launch_head_grad_reduce(a, L, st);
  if (!a->d_out) {  // only out_hidden carries gradient
    k_copy_or_zero<<<cdiv(BN * H, 256), 256, 0, st>>>(a->d_hidden, L.G, BN * H, H, L.route.g_tiled);
    REGT_LAUNCHED("k_copy_or_zero", st);
    return 0;
  }
  if (L.route.head == HeadPath::Tf32x3) return head_backward_f(a, L, st);
  HeadK k = make_headk(a, L, nullptr, nullptr);
  const int nblk = cdiv(BN, TMH);
  const size_t smem = ((size_t)TMH * (O + 1) + TMH * (HEAD_HID + 1) + KT * TN + 4) * sizeof(float);
  REGT_CUDA(cudaFuncSetAttribute(k_head_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_head_bwd<<<nblk, TMH * 4, smem, st>>>(k);
  REGT_LAUNCHED("k_head_bwd", st);
  // weight gradients: dW2 = d_out^T a1, dW1 = d_a1^T relu(hid); biases = column sums
  // split-K over the rows: enough splits to fill the SMs (partials are summed in a fixed order by k_reduce_splits)
  const int splits = (int)max(1ll, min(128ll, BN / 128));
  float* part = L.part;
  if (a->precision == REGT_PREC_TF32X3 && H % 32 == 0 && BN >= 128) {
    // dW1, db1 on the tensor cores: column 16 of the cell's feature plane is all ones, its first BN rows are the operand.
    // A head-only call ran no cell: it writes that plane itself
    if (L.route.cell == CellPath::None && launch_ones_f((int)BN, (int)((BN + 127) / 128 * 128), L.Feat, st)) return -1;
    if (launch_head_dw1_tf32x3(a, L, L.Feat, st)) return -1;
    TNBatch tb{};
    tb.nprob = 1;
    tb.p[0] = TNProb{a->d_out, L.a1, part, O, HEAD_HID, O, HEAD_HID, 0};
    if (launch_wgrad_tn(tb, BN, splits, st)) return -1;
    if (launch_reduce_splits(tb.p[0].part, a->g.head_w2, (long long)O * HEAD_HID, splits, a->accumulate, st)) return -1;
    if (launch_colsum(a->d_out, O, O, BN, splits, part, st)) return -1;
    return launch_reduce_splits(part, a->g.head_b2, O, splits, a->accumulate, st);
  }
  TNBatch tb{};
  tb.nprob = 2;
  tb.p[0] = TNProb{a->d_out, L.a1, part, O, HEAD_HID, O, HEAD_HID, 0};
  tb.p[1] = TNProb{L.d_a1, a->out_hidden, part + (size_t)splits * O * HEAD_HID, HEAD_HID, H, HEAD_HID, H, 1};
  if (launch_wgrad_tn(tb, BN, splits, st)) return -1;
  if (launch_reduce_splits(tb.p[0].part, a->g.head_w2, (long long)O * HEAD_HID, splits, a->accumulate, st)) return -1;
  if (launch_reduce_splits(tb.p[1].part, a->g.head_w1, (long long)HEAD_HID * H, splits, a->accumulate, st)) return -1;
  if (launch_colsum(a->d_out, O, O, BN, splits, part, st)) return -1;
  if (launch_reduce_splits(part, a->g.head_b2, O, splits, a->accumulate, st)) return -1;
  if (launch_colsum(L.d_a1, HEAD_HID, HEAD_HID, BN, splits, part, st)) return -1;
  if (launch_reduce_splits(part, a->g.head_b1, HEAD_HID, splits, a->accumulate, st)) return -1;
  return 0;
}

}  // namespace regt
