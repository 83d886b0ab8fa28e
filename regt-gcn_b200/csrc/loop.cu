// The callers on either side of the hot path (SURVEY 8f.1, 8f.2), on the device:
//   regt_window_gather   load_dataset.py:451-457 materialises every sliding window of node_data [N, F, T_total] on the host
//                        (T_in-fold duplication, then one H2D copy per snapshot, run.py:172).  Here node_data stays
//                        resident and a batch of windows x [B,N,F,T_in], y [B,N,T_out] is gathered by one kernel.
//   regt_rmsprop_step    run.py:145,194: torch.optim.RMSprop (alpha 0.99, eps 1e-8, weight_decay, no momentum, not centred)
//                        once per epoch over ALL parameters -- one launch over the flat parameter / gradient buffers.
//   regt_eval_metrics    predict.py:142-194: MAE, RMSE and the p95-normalised MAPE of a batch of snapshots without the
//                        per-snapshot .cpu() round trips: per-snapshot sums and numpy's linear-interpolation percentile
//                        (radix select on the float keys) on the device.  regt_eval_metrics_masked does the same over the
//                        valid targets only (a missing reading is marked by a null value or NaN, as in METR-LA / PEMS-BAY).
#include "common.cuh"

namespace regt {
namespace {

__global__ void __launch_bounds__(256) k_window_gather(const float* __restrict__ node_data, const int64_t* __restrict__ starts, int B,
                                                       int N, int Fd, long long Ttot, int T_in, int T_out, int target_f,
                                                       float* __restrict__ x, float* __restrict__ y) {
  const long long nx = (long long)B * N * Fd * T_in, ny = (long long)B * N * T_out;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < nx) {
    const int t = (int)(i % T_in);
    long long r = i / T_in;
    const int f = (int)(r % Fd);
    r /= Fd;
    const int n = (int)(r % N), b = (int)(r / N);
    x[i] = __ldg(node_data + ((size_t)n * Fd + f) * Ttot + starts[b] + t);
  } else if (i < nx + ny) {
    const long long j = i - nx;
    const int o = (int)(j % T_out);
    const long long r = j / T_out;
    const int n = (int)(r % N), b = (int)(r / N);
    y[j] = __ldg(node_data + ((size_t)n * Fd + target_f) * Ttot + starts[b] + T_in + o);
  }
}

__global__ void __launch_bounds__(256) k_rmsprop(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ sq, long long n,
                                                 float lr, float alpha, float eps, float wd) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float gi = g[i];
  if (wd != 0.f) gi = fmaf(wd, p[i], gi);                    // grad = grad + weight_decay * param
  const float s = alpha * sq[i] + (1.0f - alpha) * gi * gi;  // square_avg.mul_(alpha).addcmul_(grad, grad, value=1 - alpha)
  sq[i] = s;
  p[i] = p[i] - lr * (gi / (sqrtf(s) + eps));                // param.addcdiv_(grad, avg.sqrt().add_(eps), value=-lr)
}

// order-preserving key of a float (total order, -0 < +0)
__device__ __forceinline__ uint32_t fkey(float v) {
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float funkey(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
__device__ __forceinline__ bool valid_target(float v, float null_v) { return v == v && v != null_v; }
// k-th smallest (0-based) of v[0..n) (MASKED: of its valid entries); 4 passes of an 8-bit radix select by one block; result
// broadcast through shared memory
template <bool MASKED>
__device__ uint32_t block_select(const float* __restrict__ v, long long n, long long k, uint32_t* hist /*[256]*/, uint32_t* bc /*[2]*/,
                                 float null_v = 0.f) {
  uint32_t prefix = 0, mask = 0;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
      const float vi = v[i];
      if (MASKED && !valid_target(vi, null_v)) continue;
      const uint32_t key = fkey(vi);
      if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      long long kk = k;
      uint32_t d = 0;
      for (; d < 255; ++d) {
        if (kk < (long long)hist[d]) break;
        kk -= hist[d];
      }
      bc[0] = d;
      bc[1] = (uint32_t)kk;   // rank inside the chosen bucket (fits: bucket count <= n, n < 2^32 enforced by the launcher)
    }
    __syncthreads();
    prefix |= bc[0] << shift;
    mask |= 255u << shift;
    k = bc[1];
    __syncthreads();
  }
  return prefix;
}

// one block per snapshot b: sums[b] = { sum |y - out| , sum (y - out)^2 , p95(y_b) , sum |y - out| / p95 }
__global__ void __launch_bounds__(256) k_eval_metrics(const float* __restrict__ out, const float* __restrict__ y, long long n,
                                                      double q, double* __restrict__ sums) {
  __shared__ uint32_t hist[256], bc[2];
  __shared__ double red[2][8];
  const float* yb = y + (size_t)blockIdx.x * n;
  const float* ob = out + (size_t)blockIdx.x * n;
  // numpy.percentile(method='linear'): virtual index q/100 * (n-1), lerp between the two neighbouring order statistics
  const double pos = q / 100.0 * (double)(n - 1);
  const long long lo = (long long)floor(pos);
  const double t = pos - (double)lo;
  const float a = funkey(block_select<false>(yb, n, lo, hist, bc));
  const float b = (lo + 1 < n) ? funkey(block_select<false>(yb, n, lo + 1, hist, bc)) : a;
  const double diff = (double)b - (double)a;
  const double p95 = t >= 0.5 ? (double)b - diff * (1.0 - t) : (double)a + diff * t;   // numpy's _lerp
  double s1 = 0.0, s2 = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const float e = yb[i] - ob[i];          // fp32 difference, as (batch.y - out) in predict.py
    s1 += (double)fabsf(e);
    s2 += (double)(e * e);                  // ((batch.y - out) ** 2) is an fp32 product
  }
  for (int d = 16; d > 0; d >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, d);
    s2 += __shfl_xor_sync(0xffffffffu, s2, d);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s1;
    red[1][threadIdx.x >> 5] = s2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int w = 0; w < 8; ++w) {
      t1 += red[0][w];
      t2 += red[1][w];
    }
    double* o = sums + (size_t)blockIdx.x * 4;
    o[0] = t1;
    o[1] = t2;
    o[2] = p95;
    o[3] = t1 / (double)(float)p95;   // predict.py divides the fp32 errors by the percentile: inf / nan when it is 0
  }
}

// k_eval_metrics over the valid targets: sums[b] = { c_b, sum m|e|, sum m e^2, percentile q of the valid y_b, sum m|e| / it }
__global__ void __launch_bounds__(256) k_eval_metrics_masked(const float* __restrict__ out, const float* __restrict__ y, long long n,
                                                             double q, float null_v, double* __restrict__ sums) {
  __shared__ uint32_t hist[256], bc[2];
  __shared__ double red[2][8];
  __shared__ unsigned long long redc[8];
  __shared__ long long cnt_s;
  const float* yb = y + (size_t)blockIdx.x * n;
  const float* ob = out + (size_t)blockIdx.x * n;
  double s1 = 0.0, s2 = 0.0;
  unsigned long long c = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const float yv = yb[i];
    if (!valid_target(yv, null_v)) continue;
    const float e = yv - ob[i];
    ++c;
    s1 += (double)fabsf(e);
    s2 += (double)(e * e);
  }
  for (int d = 16; d > 0; d >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, d);
    s2 += __shfl_xor_sync(0xffffffffu, s2, d);
    c += __shfl_xor_sync(0xffffffffu, c, d);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s1;
    red[1][threadIdx.x >> 5] = s2;
    redc[threadIdx.x >> 5] = c;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < 8; ++w) t += redc[w];
    cnt_s = (long long)t;
  }
  __syncthreads();
  const long long cnt = cnt_s;
  double p = __longlong_as_double(0x7ff8000000000000ll);   // NaN: no valid target
  if (cnt > 0) {
    const double pos = q / 100.0 * (double)(cnt - 1);
    const long long lo = (long long)floor(pos);
    const double t = pos - (double)lo;
    const float a = funkey(block_select<true>(yb, n, lo, hist, bc, null_v));
    const float b = (lo + 1 < cnt) ? funkey(block_select<true>(yb, n, lo + 1, hist, bc, null_v)) : a;
    const double diff = (double)b - (double)a;
    p = t >= 0.5 ? (double)b - diff * (1.0 - t) : (double)a + diff * t;
  }
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int w = 0; w < 8; ++w) {
      t1 += red[0][w];
      t2 += red[1][w];
    }
    double* o = sums + (size_t)blockIdx.x * 5;
    o[0] = (double)cnt;
    o[1] = t1;
    o[2] = t2;
    o[3] = p;
    o[4] = cnt > 0 ? t1 / (double)(float)p : p;
  }
}
}  // namespace
}  // namespace regt

using namespace regt;

extern "C" int regt_window_gather(const float* node_data, const int64_t* starts, int32_t B, int32_t N, int32_t Fd, int64_t T_total,
                                  int32_t T_in, int32_t T_out, int32_t target_f, float* x, float* y, regt_stream_t stream) {
  REGT_CHECK(node_data && starts && x && B > 0 && N > 0 && Fd > 0 && T_in > 0 && T_out >= 0 && T_total >= T_in + T_out,
             "regt_window_gather: bad arguments");
  REGT_CHECK(T_out == 0 || (y && target_f >= 0 && target_f < Fd), "regt_window_gather: bad target feature %d", target_f);
  const long long total = (long long)B * N * Fd * T_in + (long long)B * N * T_out;
  k_window_gather<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(node_data, starts, B, N, Fd, T_total, T_in, T_out, target_f, x, y);
  REGT_LAUNCHED("k_window_gather", (cudaStream_t)stream);
  return 0;
}

extern "C" int regt_rmsprop_step(float* params, const float* grads, float* square_avg, int64_t n, float lr, float alpha, float eps,
                                 float weight_decay, regt_stream_t stream) {
  REGT_CHECK(params && grads && square_avg && n > 0, "regt_rmsprop_step: bad arguments");
  k_rmsprop<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(params, grads, square_avg, n, lr, alpha, eps, weight_decay);
  REGT_LAUNCHED("k_rmsprop", (cudaStream_t)stream);
  return 0;
}

// sums [B][4] (double, device): per snapshot sum|e|, sum e^2, percentile q of y, sum|e| / percentile
extern "C" int regt_eval_metrics(const float* out, const float* y, int32_t B, int64_t n_per_snapshot, double q, double* sums,
                                 regt_stream_t stream) {
  REGT_CHECK(out && y && sums && B > 0 && n_per_snapshot > 0 && n_per_snapshot < (1ll << 32) && q >= 0.0 && q <= 100.0,
             "regt_eval_metrics: bad arguments");
  k_eval_metrics<<<B, 256, 0, (cudaStream_t)stream>>>(out, y, n_per_snapshot, q, sums);
  REGT_LAUNCHED("k_eval_metrics", (cudaStream_t)stream);
  return 0;
}

// sums [B][5] (double, device): per snapshot valid count, sum m|e|, sum m e^2, percentile q of the valid y, sum m|e| / percentile
extern "C" int regt_eval_metrics_masked(const float* out, const float* y, int32_t B, int64_t n_per_snapshot, double q, float null_value,
                                        double* sums, regt_stream_t stream) {
  REGT_CHECK(out && y && sums && B > 0 && n_per_snapshot > 0 && n_per_snapshot < (1ll << 32) && q >= 0.0 && q <= 100.0,
             "regt_eval_metrics_masked: bad arguments");
  k_eval_metrics_masked<<<B, 256, 0, (cudaStream_t)stream>>>(out, y, n_per_snapshot, q, null_value, sums);
  REGT_LAUNCHED("k_eval_metrics_masked", (cudaStream_t)stream);
  return 0;
}
