// fp32 FFMA building blocks shared by the parity-mode (REGT_PREC_FP32) kernels.
#pragma once
#include "common.cuh"

namespace regt {

constexpr int KT = 16;  // k-chunk of the weight tile staged in shared memory
constexpr int TN = 64;  // output columns per pass (16 thread columns x 4)

// acc[i][j] += sum_k As[(ty*4+i)*lda + k] * W[k*ldw + n0 + tx*4 + j]   for k in [0,K)
// W is row-major in global memory; columns >= ncols read as 0.  Every thread of the block
// must call this (it contains __syncthreads).  Ws: shared scratch of KT*TN floats.
template <int NT>
__device__ __forceinline__ void tile_gemm(const float* As, int lda, int K, const float* __restrict__ W, int ldw,
                                          int n0, int ncols, float* Ws, float (&acc)[4][4], int ty, int tx) {
  const bool vec = ((ldw & 3) == 0) && ((ncols & 3) == 0) && ((((uintptr_t)W) & 15) == 0);
  for (int k0 = 0; k0 < K; k0 += KT) {
    __syncthreads();
    if (vec) {
      for (int i = threadIdx.x; i < KT * TN / 4; i += NT) {
        int kk = i / (TN / 4), c4 = i % (TN / 4);
        int k = k0 + kk, n = n0 + c4 * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < K && n < ncols) v = __ldg(reinterpret_cast<const float4*>(W + (size_t)k * ldw + n));
        *reinterpret_cast<float4*>(Ws + kk * TN + c4 * 4) = v;
      }
    } else {
      for (int i = threadIdx.x; i < KT * TN; i += NT) {
        int kk = i / TN, c = i % TN;
        int k = k0 + kk, n = n0 + c;
        Ws[i] = (k < K && n < ncols) ? __ldg(W + (size_t)k * ldw + n) : 0.f;
      }
    }
    __syncthreads();
    const int kmax = min(KT, K - k0);
    const float* a0 = As + (ty * 4) * lda + k0;
#pragma unroll 4
    for (int kk = 0; kk < kmax; ++kk) {
      const float4 b = *reinterpret_cast<const float4*>(Ws + kk * TN + tx * 4);
      float a[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = a0[i * lda + kk];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(a[i], b.x, acc[i][0]);
        acc[i][1] = fmaf(a[i], b.y, acc[i][1]);
        acc[i][2] = fmaf(a[i], b.z, acc[i][2]);
        acc[i][3] = fmaf(a[i], b.w, acc[i][3]);
      }
    }
  }
}

__device__ __forceinline__ void zero_acc(float (&acc)[4][4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
}

// deterministic block sum (fixed shuffle tree + fixed warp order); result valid in thread 0
__device__ __forceinline__ float block_sum(float v, float* red /* >= 32 floats */) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    for (int w = 0; w < nw; ++w) s += red[w];
  }
  return s;
}

// deterministic sum over per-CTA partials: blockDim = (32 outputs, 8 partial subsets).
// Thread (x, y) adds partials y, y+8, ... of output i; the 8 subset sums are combined in a fixed
// order.  Valid result in the threads with threadIdx.y == 0.  All threads of the block must call.
__device__ __forceinline__ float sum_parts_32x8(const float* __restrict__ part, size_t stride, int nparts, long long i,
                                                bool in_range, float (*red)[32]) {
  float s0 = 0.f, s1 = 0.f;
  if (in_range) {
    int p = threadIdx.y;
    for (; p + 8 < nparts; p += 16) {
      s0 += __ldg(part + (size_t)p * stride + i);
      s1 += __ldg(part + (size_t)(p + 8) * stride + i);
    }
    if (p < nparts) s0 += __ldg(part + (size_t)p * stride + i);
  }
  red[threadIdx.y][threadIdx.x] = s0 + s1;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.y == 0) {
#pragma unroll
    for (int y = 0; y < 8; ++y) s += red[y][threadIdx.x];
  }
  return s;
}

// ---- split-K "TN" GEMM:  C[m][n] = sum_r A[r*lda + m] * B[r*ldb + n]  (weight gradients) ----
struct TNProb {
  const float* A;
  const float* B;
  float* part;  // [splits][M][N]
  int lda, ldb, M, N;
  int relu_b;   // apply max(.,0) to B on load
};
struct TNBatch {
  TNProb p[3];
  int nprob;
};

}  // namespace regt
