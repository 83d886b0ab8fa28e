// Time steps shared across the sliding windows of an epoch (include/regt_b200.h, regt_combine_*; regt_b200/loop.py).
//
// The hidden state is not carried across periods (DESIGN section 2): the cell output of period t of a window is a function
// of that period's input alone, so with H'(tau) the cell output of time step tau,
//   out_hidden[w] = sum_{t<T} p_t H'(w + t)                                  p = softmax(attention)
// and the gradients regroup the same way:
//   G'(tau)  = sum_{t : 0 <= tau - t < C} p_t G[tau - t]                      (what the cell backward of step tau needs)
//   dprobs_t = sum_w <G[w], H'(w + t)>,   d attention = p (dprobs - <p, dprobs>)
// Both kernels are HBM-bound streams along tau: a thread owns four columns of the N*H-wide rows and keeps the last T rows
// it needs in shared memory (its own slots only: no barrier inside the stream), so every element of H' and G is read once
// when the columns fill the device.  A narrower pass is split into chunks along tau; a chunk re-reads the T - 1 rows
// before it.  Sums run in period order; the attention-gradient terms are fp64 per thread, then summed over the threads of
// a block and over the blocks in a fixed order (the softmax Jacobian takes differences of nearly equal sums).
#include "common.cuh"

namespace regt {
namespace {

constexpr int CB_PF = 4;              // rows each thread loads before it uses them (bytes in flight)
constexpr int CB_MAX_T = 256;         // periods: a thread keeps T float4 ring slots and T fp64 sums in shared memory
constexpr int CB_MAX_BLOCKS = 1184;   // blocks of the persistent grids (and fp64 partial rows of the backward)

__device__ __forceinline__ void fma4(float p, const float4& v, float4& acc) {
  acc.x = fmaf(p, v.x, acc.x);
  acc.y = fmaf(p, v.y, acc.y);
  acc.z = fmaf(p, v.z, acc.z);
  acc.w = fmaf(p, v.w, acc.w);
}

// out[w] = sum_t p_t Hs[w + t] for the windows [w0, w1) of each chunk; ring slot of row r is r % T
__global__ void __launch_bounds__(128) k_comb_fwd(const float* __restrict__ att, const float4* __restrict__ Hs, int C, int T,
                                                  long long w4, int wchunk, int nchunk, float4* __restrict__ out) {
  extern __shared__ float4 ring[];   // [T][blockDim.x]
  __shared__ float p[CB_MAX_T];
  if (threadIdx.x == 0) attention_softmax(att, T, p);
  __syncthreads();
  const int nt = blockDim.x, me = threadIdx.x;
  const long long ntile = (w4 + nt - 1) / nt;
  for (long long item = blockIdx.x; item < ntile * nchunk; item += gridDim.x) {
    const long long j = (item % ntile) * nt + me;
    const int w0 = (int)(item / ntile) * wchunk, w1 = min(C, w0 + wchunk), r1 = w1 + T - 1;
    if (j >= w4) continue;
    for (int base = w0; base < r1; base += CB_PF) {
      float4 v[CB_PF];
#pragma unroll
      for (int k = 0; k < CB_PF; ++k) v[k] = base + k < r1 ? __ldg(Hs + (size_t)(base + k) * w4 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < CB_PF; ++k) {
        const int tau = base + k;
        if (tau >= r1) break;
        ring[(size_t)(tau % T) * nt + me] = v[k];
        const int w = tau - T + 1;
        if (w < w0) continue;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int slot = w % T;
        for (int t = 0; t < T; ++t) {
          fma4(p[t], ring[(size_t)slot * nt + me], acc);
          if (++slot == T) slot = 0;
        }
        out[(size_t)w * w4 + j] = acc;
      }
    }
  }
}

// Gs[tau] = sum_t p_t G[tau - t] for the steps [s0, s1) of each chunk (G rows outside [0, C) are zeros), and this thread's
// share of dprobs_t = sum <G[tau - t], Hs[tau]>; part[block][t] = the block's fp64 sums
__global__ void __launch_bounds__(128) k_comb_bwd(const float* __restrict__ att, const float4* __restrict__ Hs, const float4* __restrict__ G,
                                                  int S, int C, int T, long long w4, int schunk, int nchunk, float4* __restrict__ Gs,
                                                  double* __restrict__ part) {
  extern __shared__ float4 sm[];
  const int nt = blockDim.x, me = threadIdx.x;
  float4* ring = sm;                                      // [T][nt]  G rows tau-T+1 .. tau, slot r % T
  double* dp = reinterpret_cast<double*>(sm + (size_t)T * nt);   // [T][nt]
  __shared__ float p[CB_MAX_T];
  for (int t = 0; t < T; ++t) dp[(size_t)t * nt + me] = 0.0;
  if (me == 0) attention_softmax(att, T, p);
  __syncthreads();
  const long long ntile = (w4 + nt - 1) / nt;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long item = blockIdx.x; item < ntile * nchunk; item += gridDim.x) {
    const long long j = (item % ntile) * nt + me;
    const int s0 = (int)(item / ntile) * schunk, s1 = min(S, s0 + schunk);
    if (j >= w4) continue;
    for (int r = s0 - T + 1; r < s0; ++r)   // the rows before the chunk that its first steps combine
      ring[(size_t)((r % T + T) % T) * nt + me] = (r >= 0 && r < C) ? __ldg(G + (size_t)r * w4 + j) : zero;
    for (int base = s0; base < s1; base += CB_PF) {
      float4 g[CB_PF], h[CB_PF];
#pragma unroll
      for (int k = 0; k < CB_PF; ++k) {
        const int tau = base + k;
        g[k] = tau < min(s1, C) ? __ldg(G + (size_t)tau * w4 + j) : zero;
        h[k] = tau < s1 ? __ldg(Hs + (size_t)tau * w4 + j) : zero;
      }
#pragma unroll
      for (int k = 0; k < CB_PF; ++k) {
        const int tau = base + k;
        if (tau >= s1) break;
        int slot = tau % T;
        ring[(size_t)slot * nt + me] = g[k];
        float4 acc = zero;
        for (int t = 0; t < T; ++t) {   // G[tau - t] sits in slot (tau - t) % T
          const float4 gv = ring[(size_t)slot * nt + me];
          fma4(p[t], gv, acc);
          float d = gv.x * h[k].x;
          d = fmaf(gv.y, h[k].y, d);
          d = fmaf(gv.z, h[k].z, d);
          d = fmaf(gv.w, h[k].w, d);
          dp[(size_t)t * nt + me] += (double)d;
          if (--slot < 0) slot = T - 1;
        }
        Gs[(size_t)tau * w4 + j] = acc;
      }
    }
  }
  __syncthreads();
  for (int t = me; t < T; t += nt) {   // threads of the block in order
    double s = 0.0;
    for (int i = 0; i < nt; ++i) s += dp[(size_t)t * nt + i];
    part[(size_t)blockIdx.x * T + t] = s;
  }
}

// dprobs_t = sum of the blocks' partials in block order; attention_grad[t] += p_t (dprobs_t - sum_s p_s dprobs_s)
__global__ void k_comb_attn(const float* __restrict__ att, const double* __restrict__ part, int nparts, int T, float* __restrict__ grad) {
  __shared__ float p[CB_MAX_T];
  __shared__ double dpr[CB_MAX_T];
  if (threadIdx.x == 0) attention_softmax(att, T, p);
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    double s = 0.0;
    for (int b = 0; b < nparts; ++b) s += part[(size_t)b * T + t];
    dpr[t] = s;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    double dot = 0.0;
    for (int s = 0; s < T; ++s) dot += (double)p[s] * dpr[s];
    grad[t] += (float)((double)p[t] * (dpr[t] - dot));
  }
}

// threads per block: a thread keeps T ring slots (16 B) and T fp64 sums (8 B) in shared memory
int comb_threads(int T) {
  int nt = 128;
  while (nt > 32 && (size_t)nt * T * 24 > 200 * 1024) nt >>= 1;
  return nt;
}

// persistent grid over (column tile, chunk) items: chunks along tau only when the column tiles alone leave SMs idle
template <typename K>
int comb_grid(K kern, int nt, size_t smem, long long w4, int rows, int T, int* chunk, int* nchunk) {
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nt, smem) != cudaSuccess || occ < 1) occ = 1;
  const long long ntile = (w4 + nt - 1) / nt, resident = (long long)sm_count() * occ;
  long long nc = ntile >= resident ? 1 : min((long long)(rows + T - 1) / T, (2 * resident + ntile - 1) / ntile);
  nc = max(1ll, nc);
  *chunk = (int)((rows + nc - 1) / nc);
  *nchunk = (rows + *chunk - 1) / *chunk;
  return (int)min(min(ntile * *nchunk, resident), (long long)CB_MAX_BLOCKS);
}

int check_sizes(const char* who, const float* att, const float* Hs, int S, int C, int T, long long width) {
  REGT_CHECK(att && Hs, "%s: attention / Hs is NULL", who);
  REGT_CHECK(T >= 1 && T <= CB_MAX_T, "%s: T=%d periods must be in 1..%d", who, T, CB_MAX_T);
  REGT_CHECK(C >= 1, "%s: C=%d windows must be >= 1", who, C);
  REGT_CHECK((long long)S == (long long)C + T - 1, "%s: S=%d steps must be C + T - 1 = %lld (C=%d windows of T=%d periods)", who,
             S, (long long)C + T - 1, C, T);
  REGT_CHECK(width > 0 && width % 4 == 0, "%s: width=%lld must be a positive multiple of 4 (N*H)", who, width);
  REGT_CHECK(((uintptr_t)Hs & 15) == 0, "%s: Hs must be 16-byte aligned", who);
  return 0;
}

}  // namespace
}  // namespace regt

using namespace regt;

extern "C" size_t regt_combine_scratch_bytes(int32_t T) { return T >= 1 ? (size_t)CB_MAX_BLOCKS * T * sizeof(double) : 0; }

extern "C" int regt_combine_forward(const float* attention, const float* Hs, int32_t S, int32_t C, int32_t T, int64_t width,
                                    float* out_hidden, regt_stream_t stream) {
  if (check_sizes("regt_combine_forward", attention, Hs, S, C, T, width)) return -1;
  REGT_CHECK(out_hidden && ((uintptr_t)out_hidden & 15) == 0, "regt_combine_forward: out_hidden is NULL or not 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int nt = comb_threads(T);
  const size_t smem = (size_t)T * nt * sizeof(float4);
  REGT_CUDA(cudaFuncSetAttribute(k_comb_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int chunk = 0, nchunk = 0;
  const int grid = comb_grid(k_comb_fwd, nt, smem, width / 4, C, T, &chunk, &nchunk);
  prof_mark("<begin>", st);
  k_comb_fwd<<<grid, nt, smem, st>>>(attention, reinterpret_cast<const float4*>(Hs), C, T, width / 4, chunk, nchunk,
                                     reinterpret_cast<float4*>(out_hidden));
  REGT_LAUNCHED("k_comb_fwd", st);
  return 0;
}

extern "C" int regt_combine_backward(const float* attention, const float* Hs, const float* G, int32_t S, int32_t C, int32_t T,
                                     int64_t width, float* Gs, float* attention_grad, void* scratch, size_t scratch_bytes,
                                     regt_stream_t stream) {
  if (check_sizes("regt_combine_backward", attention, Hs, S, C, T, width)) return -1;
  REGT_CHECK(G && Gs && ((uintptr_t)G & 15) == 0 && ((uintptr_t)Gs & 15) == 0,
             "regt_combine_backward: G / Gs is NULL or not 16-byte aligned");
  REGT_CHECK(scratch && scratch_bytes >= regt_combine_scratch_bytes(T) && ((uintptr_t)scratch & 7) == 0,
             "regt_combine_backward: scratch missing, too small (%zu < %zu bytes) or not 8-byte aligned", scratch_bytes,
             regt_combine_scratch_bytes(T));
  cudaStream_t st = (cudaStream_t)stream;
  const int nt = comb_threads(T);
  const size_t smem = (size_t)T * nt * (sizeof(float4) + sizeof(double));
  REGT_CUDA(cudaFuncSetAttribute(k_comb_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int chunk = 0, nchunk = 0;
  const int grid = comb_grid(k_comb_bwd, nt, smem, width / 4, S, T, &chunk, &nchunk);
  double* part = static_cast<double*>(scratch);
  prof_mark("<begin>", st);
  k_comb_bwd<<<grid, nt, smem, st>>>(attention, reinterpret_cast<const float4*>(Hs), reinterpret_cast<const float4*>(G), S, C, T,
                                     width / 4, chunk, nchunk, reinterpret_cast<float4*>(Gs), part);
  REGT_LAUNCHED("k_comb_bwd", st);
  if (attention_grad) {
    k_comb_attn<<<1, 256, 0, st>>>(attention, part, grid, T, attention_grad);
    REGT_LAUNCHED("k_comb_attn", st);
  }
  return 0;
}
