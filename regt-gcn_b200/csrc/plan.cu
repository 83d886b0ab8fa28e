// K1: static-graph plan.  edge_index (COO, int64) -> CSR by destination with the
// normalised operator values, once per static graph.
//
//   regt_gcn_plan_build  : PyG gcn_norm semantics (SURVEY Appendix A.1) -- the reference
//                          recomputes this 3*T times per sample (models/utils.py:169,175,181)
//   regt_cheb_plan_build : PyG get_laplacian('sym') + Chebyshev rescale (Appendix A.3) --
//                          recomputed R*T times per sample (models/RegionalTemporalGCN.py:136-140)
//
// Determinism: all floating-point sums run sequentially in the canonical (input) order,
// so degrees and values are reproducible bit for bit; integer structures are exact.
// Sorting strategy: histogram -> scan -> atomic-cursor placement -> per-slot rank by the
// unique entry id (any placement order gives the same canonical result).
#include "common.cuh"

namespace regt {

// ---------------- single-block exclusive scan (plan build is off the hot loop) ---------
__global__ void k_exclusive_scan(const int32_t* __restrict__ in, int32_t* __restrict__ out, int n,
                                 int32_t* __restrict__ total) {
  __shared__ int32_t warp_sums[32];
  __shared__ int32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + threadIdx.x;
    int32_t v = i < n ? in[i] : 0;
    int32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int32_t w = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0;
      int32_t wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        int32_t t = __shfl_up_sync(0xffffffffu, wi, d);
        if (lane >= d) wi += t;
      }
      warp_sums[lane] = wi - w;  // exclusive prefix of warp sums
    }
    __syncthreads();
    int32_t carry = carry_s;
    if (i < n) out[i] = carry + warp_sums[wid] + incl - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = carry + warp_sums[wid] + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0 && total) *total = carry_s;
}

static int exclusive_scan(const int32_t* in, int32_t* out, int n, int32_t* total, cudaStream_t st) {
  k_exclusive_scan<<<1, 1024, 0, st>>>(in, out, n, total);
  REGT_LAUNCH_CHECK();
  return 0;
}

// ---------------- generic: bucket entries by key, canonical order inside a bucket ------
__global__ void k_count_keys(const int32_t* __restrict__ key, int n, int32_t* __restrict__ cnt) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&cnt[key[i]], 1);
}
__global__ void k_place(const int32_t* __restrict__ key, int n, const int32_t* __restrict__ ptr,
                        int32_t* __restrict__ cursor, int32_t* __restrict__ tmp) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    int k = key[i];
    tmp[ptr[k] + atomicAdd(&cursor[k], 1)] = i;
  }
}
// every slot finds its rank among the entry ids of its bucket
__global__ void k_rank(const int32_t* __restrict__ key, const int32_t* __restrict__ ptr,
                       const int32_t* __restrict__ tmp, int n, int32_t* __restrict__ sorted) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  int id = tmp[s];
  int k = key[id];
  int b = ptr[k], e = ptr[k + 1], r = 0;
  for (int j = b; j < e; ++j) r += tmp[j] < id;
  sorted[b + r] = id;
}

// key[n] -> ptr[nb+1], sorted[n] (entry ids grouped by key, ascending id inside a group)
static int bucket_sort(const int32_t* key, int n, int nb, int32_t* ptr, int32_t* sorted, int32_t* cnt_scratch,
                       int32_t* tmp_scratch, cudaStream_t st) {
  REGT_CUDA(cudaMemsetAsync(cnt_scratch, 0, sizeof(int32_t) * (nb + 1), st));
  if (n > 0) {
    k_count_keys<<<cdiv(n, 256), 256, 0, st>>>(key, n, cnt_scratch);
    REGT_LAUNCH_CHECK();
  }
  if (exclusive_scan(cnt_scratch, ptr, nb + 1, nullptr, st)) return -1;
  REGT_CUDA(cudaMemsetAsync(cnt_scratch, 0, sizeof(int32_t) * (nb + 1), st));
  if (n > 0) {
    k_place<<<cdiv(n, 256), 256, 0, st>>>(key, n, ptr, cnt_scratch, tmp_scratch);
    REGT_LAUNCH_CHECK();
    k_rank<<<cdiv(n, 256), 256, 0, st>>>(key, ptr, tmp_scratch, n, sorted);
    REGT_LAUNCH_CHECK();
  }
  return 0;
}

// ---------------- gcn_norm ---------------------------------------------------------------
__global__ void k_mark_noloop(const int64_t* __restrict__ ei, int64_t E, int32_t* __restrict__ keep) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < E) keep[e] = ei[e] != ei[E + e];
}
// last self-loop edge (input order) of every node: "duplicates: last wins"
__global__ void k_last_loop(const int64_t* __restrict__ ei, int64_t E, int32_t* __restrict__ last_loop) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < E && ei[e] == ei[E + e]) atomicMax(&last_loop[ei[e]], (int32_t)e);
}
// post-normalisation entry list: kept edges at pos[e], then N loops
__global__ void k_gcn_entries(const int64_t* __restrict__ ei, const float* __restrict__ ew, int64_t E, int N,
                              const int32_t* __restrict__ keep, const int32_t* __restrict__ pos, int Ep,
                              const int32_t* __restrict__ last_loop, int32_t* __restrict__ src,
                              int32_t* __restrict__ dst, float* __restrict__ w) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < E) {
    if (keep[i]) {
      int j = pos[i];
      src[j] = (int32_t)ei[i];
      dst[j] = (int32_t)ei[E + i];
      w[j] = ew ? ew[i] : 1.0f;
    }
  } else if (i < E + N) {
    int n = (int)(i - E);
    int j = Ep + n;
    src[j] = n;
    dst[j] = n;
    int ll = last_loop[n];
    w[j] = (ew && ll >= 0) ? ew[ll] : 1.0f;
  }
}
// degree = sequential sum over the canonical row; dis = deg^-1/2 with inf -> 0
__global__ void k_row_degree(const int32_t* __restrict__ ptr, const int32_t* __restrict__ sorted,
                             const float* __restrict__ w, int N, float* __restrict__ dis) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float d = 0.f;
  for (int k = ptr[n]; k < ptr[n + 1]; ++k) d += w[sorted[k]];
  float r = 1.0f / sqrtf(d);
  dis[n] = isinf(r) ? 0.f : r;
}
__global__ void k_gcn_values(const int32_t* __restrict__ sorted, const int32_t* __restrict__ src,
                             const int32_t* __restrict__ dst, const float* __restrict__ w,
                             const float* __restrict__ dis, int nnz, int32_t* __restrict__ col,
                             float* __restrict__ val, int32_t* __restrict__ eid) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  int j = sorted[k];
  int s = src[j];
  col[k] = s;
  val[k] = dis[s] * w[j] * dis[dst[j]];
  if (eid) eid[k] = j;
}

// ---------------- cheb ---------------------------------------------------------------------
__global__ void k_cheb_entries(const int64_t* __restrict__ ei, const float* __restrict__ ew, int64_t E,
                               const int32_t* __restrict__ keep, const int32_t* __restrict__ pos,
                               const int64_t* __restrict__ list_ptr, int R, int32_t* __restrict__ src,
                               int32_t* __restrict__ dst, int32_t* __restrict__ reg, float* __restrict__ w,
                               int32_t* __restrict__ region_of) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  int lo = 0, hi = R;  // list_ptr[lo] <= e < list_ptr[hi]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (list_ptr[mid] <= e) lo = mid; else hi = mid;
  }
  int r = lo;
  int s = (int)ei[e], d = (int)ei[E + e];
  if (keep[e]) {
    int j = pos[e];
    src[j] = s; dst[j] = d; reg[j] = r;
    w[j] = ew ? ew[e] : 1.0f;
  }
  // node -> region map from every endpoint (self-loops included)
  for (int t = 0; t < 2; ++t) {
    int n = t ? d : s;
    int old = atomicCAS(&region_of[n], -1, r);
    if (old != -1 && old != r && old != -2) atomicExch(&region_of[n], -2);
  }
}
// source degree of entry j inside its own regional list: sequential over the by-source bucket
__global__ void k_cheb_dis(const int32_t* __restrict__ sptr, const int32_t* __restrict__ ssorted,
                           const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                           const int32_t* __restrict__ reg, const float* __restrict__ w, int nnz,
                           float* __restrict__ dis_src, float* __restrict__ dis_dst) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nnz) return;
  int r = reg[j];
  for (int t = 0; t < 2; ++t) {
    int node = t ? dst[j] : src[j];
    float d = 0.f;
    for (int k = sptr[node]; k < sptr[node + 1]; ++k) {
      int jj = ssorted[k];
      if (reg[jj] == r) d += w[jj];
    }
    float v = 1.0f / sqrtf(d);
    v = isinf(v) ? 0.f : v;
    if (t) dis_dst[j] = v; else dis_src[j] = v;
  }
}
__global__ void k_cheb_values(const int32_t* __restrict__ sorted, const int32_t* __restrict__ src,
                              const int32_t* __restrict__ reg, const float* __restrict__ w,
                              const float* __restrict__ dis_src, const float* __restrict__ dis_dst, int nnz,
                              int32_t* __restrict__ col, float* __restrict__ val, int32_t* __restrict__ oreg,
                              int32_t* __restrict__ eid) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  int j = sorted[k];
  col[k] = src[j];
  oreg[k] = reg[j];
  float lap = -(dis_src[j] * w[j] * dis_dst[j]);  // off-diagonal of I - D^-1/2 A D^-1/2
  lap = (2.0f * lap) / 2.0f;                       // Chebyshev rescale with lambda_max = 2
  val[k] = isinf(lap) ? 0.f : lap;
  if (eid) eid[k] = j;
}
__global__ void k_seg_flags(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ sorted,
                            const int32_t* __restrict__ dst, const int32_t* __restrict__ oreg, int nnz,
                            int32_t* __restrict__ flag) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  int n = dst[sorted[k]];
  flag[k] = (k == rowptr[n]) || (oreg[k] != oreg[k - 1]);
}
__global__ void k_seg_fill(const int32_t* __restrict__ flag, const int32_t* __restrict__ segid,
                           const int32_t* __restrict__ sorted, const int32_t* __restrict__ dst,
                           const int32_t* __restrict__ oreg, int nnz, const int32_t* __restrict__ nseg,
                           int32_t* __restrict__ seg_eptr, int32_t* __restrict__ seg_reg,
                           int32_t* __restrict__ seg_node) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) seg_eptr[*nseg] = nnz;
  if (k >= nnz) return;
  if (flag[k]) {
    int s = segid[k];
    seg_eptr[s] = k;
    seg_reg[s] = oreg[k];
    seg_node[s] = dst[sorted[k]];
  }
}
__global__ void k_seg_ptr(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ segid, int N, int nnz,
                          const int32_t* __restrict__ nseg, int32_t* __restrict__ seg_ptr) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n > N) return;
  int k = rowptr[n];
  seg_ptr[n] = (k < nnz) ? segid[k] : *nseg;
}

// ---------------- transposed operator of the input gradient (regt_xgrad_plan) ---------------
// row_of[e] = i for every entry e in [ptr[i], ptr[i+1]): destination row of an A_hat entry, segment of a regional entry
__global__ void k_row_of(const int32_t* __restrict__ ptr, int n, int32_t* __restrict__ row_of) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int e = ptr[i]; e < ptr[i + 1]; ++e) row_of[e] = i;
}
// entry ids: [0, N) identity, [N, N + ng) A_hat entries, then the regional entries; key = the input node they read
__global__ void k_xg_keys(int N, int ng, int nc, const int32_t* __restrict__ g_col, const int32_t* __restrict__ c_col,
                          int32_t* __restrict__ key) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N + ng + nc) return;
  key[i] = i < N ? i : (i < N + ng ? g_col[i - N] : c_col[i - N - ng]);
}
__global__ void k_xg_fill(const int32_t* __restrict__ sorted, int N, int ng, int nc, const int32_t* __restrict__ g_dst,
                          const float* __restrict__ g_val, const int32_t* __restrict__ c_seg, const float* __restrict__ c_val,
                          int32_t* __restrict__ col, float* __restrict__ val) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= N + ng + nc) return;
  const int id = sorted[k];
  if (id < N) {
    col[k] = id;
    val[k] = 1.0f;
  } else if (id < N + ng) {
    col[k] = N + g_dst[id - N];
    val[k] = g_val[id - N];
  } else {
    col[k] = 2 * N + c_seg[id - N - ng];
    val[k] = c_val[id - N - ng];
  }
}

}  // namespace regt

using namespace regt;

extern "C" size_t regt_xgrad_plan_workspace_bytes(const regt_graph_plan* p) {
  if (!p) return 0;
  const size_t n = (size_t)p->N + p->nnz_gcn + p->nnz_cheb;
  return 3 * align_up(n * 4, 256) + align_up((size_t)(p->N + 1) * 4, 256) + align_up((size_t)p->nnz_gcn * 4 + 4, 256) +
         align_up((size_t)p->nnz_cheb * 4 + 4, 256) + 256;
}

extern "C" int regt_xgrad_plan_build(const regt_graph_plan* p, int32_t* rowptr, int32_t* col, float* val, void* workspace,
                                     size_t workspace_bytes, regt_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  REGT_CHECK(p && rowptr && col && val, "xgrad_plan: NULL argument");
  REGT_CHECK(p->N > 0 && p->nnz_gcn >= 0 && p->nnz_cheb >= 0 && p->nseg >= 0 &&
                 (long long)p->N + p->nnz_gcn + p->nnz_cheb < (1ll << 31) && 2ll * p->N + p->nseg < (1ll << 31),
             "xgrad_plan: bad sizes");
  REGT_CHECK(p->nnz_gcn == 0 || (p->g_rowptr && p->g_col && p->g_val), "xgrad_plan: gcn CSR missing");
  REGT_CHECK(p->nnz_cheb == 0 || (p->seg_eptr && p->c_col && p->c_val), "xgrad_plan: regional CSR missing");
  REGT_CHECK(workspace && workspace_bytes >= regt_xgrad_plan_workspace_bytes(p), "xgrad_plan: workspace too small");
  const int N = p->N, ng = p->nnz_gcn, nc = p->nnz_cheb, n = N + ng + nc;
  Carver c(workspace);
  int32_t* key = c.take<int32_t>(n);
  int32_t* tmp = c.take<int32_t>(n);
  int32_t* sorted = c.take<int32_t>(n);
  int32_t* cnt = c.take<int32_t>(N + 1);
  int32_t* g_dst = c.take<int32_t>(ng + 1);
  int32_t* c_seg = c.take<int32_t>(nc + 1);
  if (ng > 0) {
    k_row_of<<<cdiv(N, 256), 256, 0, st>>>(p->g_rowptr, N, g_dst);
    REGT_LAUNCH_CHECK();
  }
  if (nc > 0) {
    k_row_of<<<cdiv(p->nseg, 256), 256, 0, st>>>(p->seg_eptr, p->nseg, c_seg);
    REGT_LAUNCH_CHECK();
  }
  k_xg_keys<<<cdiv(n, 256), 256, 0, st>>>(N, ng, nc, p->g_col, p->c_col, key);
  REGT_LAUNCH_CHECK();
  // stable by entry id: identity, then A_hat entries, then regional entries, each in canonical CSR order
  if (bucket_sort(key, n, N, rowptr, sorted, cnt, tmp, st)) return -1;
  k_xg_fill<<<cdiv(n, 256), 256, 0, st>>>(sorted, N, ng, nc, g_dst, p->g_val, c_seg, p->c_val, col, val);
  REGT_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t regt_plan_workspace_bytes(int64_t N, int64_t E) {
  // generous: ~16 int32/float arrays of (E+N) entries + a few of N
  size_t n = (size_t)(E + N + 8);
  return 20 * align_up(n * 4, 256) + 8 * align_up((size_t)(N + 8) * 4, 256) + (1 << 20);
}

extern "C" int regt_gcn_plan_build(const int64_t* edge_index, const float* edge_weight, int64_t E, int64_t N,
                                   int32_t* rowptr, int32_t* col, float* val, int32_t* eid, int32_t* nnz_out,
                                   void* workspace, size_t workspace_bytes, regt_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  REGT_CHECK(N > 0 && E >= 0 && E + N < (1ll << 31), "gcn_plan: bad sizes N=%lld E=%lld", (long long)N, (long long)E);
  REGT_CHECK(workspace_bytes >= regt_plan_workspace_bytes(N, E), "gcn_plan: workspace too small");
  Carver c(workspace);
  const int n = (int)N;
  int32_t* keep = c.take<int32_t>(E + 1);
  int32_t* pos = c.take<int32_t>(E + 1);
  int32_t* last_loop = c.take<int32_t>(N);
  int32_t* src = c.take<int32_t>(E + N);
  int32_t* dst = c.take<int32_t>(E + N);
  float* w = c.take<float>(E + N);
  int32_t* cnt = c.take<int32_t>(N + 1);
  int32_t* tmp = c.take<int32_t>(E + N);
  int32_t* sorted = c.take<int32_t>(E + N);
  float* dis = c.take<float>(N);
  int32_t* d_total = c.take<int32_t>(1);

  REGT_CUDA(cudaMemsetAsync(keep, 0, sizeof(int32_t) * (E + 1), st));
  REGT_CUDA(cudaMemsetAsync(last_loop, 0xff, sizeof(int32_t) * N, st));
  if (E > 0) {
    k_mark_noloop<<<cdiv(E, 256), 256, 0, st>>>(edge_index, E, keep);
    REGT_LAUNCH_CHECK();
    k_last_loop<<<cdiv(E, 256), 256, 0, st>>>(edge_index, E, last_loop);
    REGT_LAUNCH_CHECK();
  }
  if (exclusive_scan(keep, pos, (int)E + 1, nullptr, st)) return -1;
  int32_t Ep = 0;
  REGT_CUDA(cudaMemcpyAsync(&Ep, pos + E, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  REGT_CUDA(cudaStreamSynchronize(st));
  const int nnz = Ep + n;
  k_gcn_entries<<<cdiv(E + N, 256), 256, 0, st>>>(edge_index, edge_weight, E, n, keep, pos, Ep, last_loop, src, dst, w);
  REGT_LAUNCH_CHECK();
  if (bucket_sort(dst, nnz, n, rowptr, sorted, cnt, tmp, st)) return -1;
  k_row_degree<<<cdiv(n, 128), 128, 0, st>>>(rowptr, sorted, w, n, dis);
  REGT_LAUNCH_CHECK();
  k_gcn_values<<<cdiv(nnz, 256), 256, 0, st>>>(sorted, src, dst, w, dis, nnz, col, val, eid);
  REGT_LAUNCH_CHECK();
  (void)d_total;
  REGT_CUDA(cudaStreamSynchronize(st));
  if (nnz_out) *nnz_out = nnz;
  return 0;
}

extern "C" int regt_cheb_plan_build(const int64_t* edge_index, const float* edge_weight, const int64_t* list_ptr,
                                    int32_t R, int64_t E, int64_t N, int32_t* rowptr, int32_t* col, float* val,
                                    int32_t* reg, int32_t* eid, int32_t* seg_ptr, int32_t* seg_eptr,
                                    int32_t* seg_reg, int32_t* seg_node, int32_t* rseg_ptr, int32_t* rseg_list,
                                    int32_t* region_of, int32_t* counts_out, void* workspace,
                                    size_t workspace_bytes, regt_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  REGT_CHECK(N > 0 && E >= 0 && R >= 1 && E + N < (1ll << 31), "cheb_plan: bad sizes");
  REGT_CHECK(workspace_bytes >= regt_plan_workspace_bytes(N, E), "cheb_plan: workspace too small");
  REGT_CHECK(list_ptr[0] == 0 && list_ptr[R] == E, "cheb_plan: list_ptr must span [0,E]");
  Carver c(workspace);
  const int n = (int)N;
  int32_t* keep = c.take<int32_t>(E + 1);
  int32_t* pos = c.take<int32_t>(E + 1);
  int32_t* src = c.take<int32_t>(E + 1);
  int32_t* dst = c.take<int32_t>(E + 1);
  int32_t* ereg = c.take<int32_t>(E + 1);
  float* w = c.take<float>(E + 1);
  int32_t* cnt = c.take<int32_t>(N + 1);
  int32_t* tmp = c.take<int32_t>(E + 1);
  int32_t* sptr = c.take<int32_t>(N + 1);
  int32_t* ssorted = c.take<int32_t>(E + 1);
  int32_t* sorted = c.take<int32_t>(E + 1);
  float* dis_src = c.take<float>(E + 1);
  float* dis_dst = c.take<float>(E + 1);
  int32_t* flag = c.take<int32_t>(E + 1);
  int32_t* segid = c.take<int32_t>(E + 1);
  int32_t* d_nseg = c.take<int32_t>(1);
  int64_t* d_list = c.take<int64_t>(R + 1);

  REGT_CUDA(cudaMemcpyAsync(d_list, list_ptr, sizeof(int64_t) * (R + 1), cudaMemcpyHostToDevice, st));
  REGT_CUDA(cudaMemsetAsync(keep, 0, sizeof(int32_t) * (E + 1), st));
  REGT_CUDA(cudaMemsetAsync(region_of, 0xff, sizeof(int32_t) * N, st));
  if (E > 0) {
    k_mark_noloop<<<cdiv(E, 256), 256, 0, st>>>(edge_index, E, keep);
    REGT_LAUNCH_CHECK();
  }
  if (exclusive_scan(keep, pos, (int)E + 1, nullptr, st)) return -1;
  int32_t nnz = 0;
  REGT_CUDA(cudaMemcpyAsync(&nnz, pos + E, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  REGT_CUDA(cudaStreamSynchronize(st));
  if (E > 0) {
    k_cheb_entries<<<cdiv(E, 256), 256, 0, st>>>(edge_index, edge_weight, E, keep, pos, d_list, R, src, dst, ereg, w,
                                                 region_of);
    REGT_LAUNCH_CHECK();
  }
  // by-source buckets -> per-list source degrees
  if (bucket_sort(src, nnz, n, sptr, ssorted, cnt, tmp, st)) return -1;
  if (nnz > 0) {
    k_cheb_dis<<<cdiv(nnz, 256), 256, 0, st>>>(sptr, ssorted, src, dst, ereg, w, nnz, dis_src, dis_dst);
    REGT_LAUNCH_CHECK();
  }
  // by-destination CSR
  if (bucket_sort(dst, nnz, n, rowptr, sorted, cnt, tmp, st)) return -1;
  int32_t nseg = 0;
  if (nnz > 0) {
    k_cheb_values<<<cdiv(nnz, 256), 256, 0, st>>>(sorted, src, ereg, w, dis_src, dis_dst, nnz, col, val, reg, eid);
    REGT_LAUNCH_CHECK();
    k_seg_flags<<<cdiv(nnz, 256), 256, 0, st>>>(rowptr, sorted, dst, reg, nnz, flag);
    REGT_LAUNCH_CHECK();
    if (exclusive_scan(flag, segid, nnz, d_nseg, st)) return -1;
    k_seg_fill<<<cdiv(nnz, 256), 256, 0, st>>>(flag, segid, sorted, dst, reg, nnz, d_nseg, seg_eptr, seg_reg, seg_node);
    REGT_LAUNCH_CHECK();
    k_seg_ptr<<<cdiv(n + 1, 256), 256, 0, st>>>(rowptr, segid, n, nnz, d_nseg, seg_ptr);
    REGT_LAUNCH_CHECK();
    REGT_CUDA(cudaMemcpyAsync(&nseg, d_nseg, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    REGT_CUDA(cudaStreamSynchronize(st));
    // segments grouped by region (ascending segment id inside a region) for the per-region wgrad
    int32_t* cnt_r = c.take<int32_t>(R + 1);
    if (bucket_sort(seg_reg, nseg, R, rseg_ptr, rseg_list, cnt_r, tmp, st)) return -1;
  } else {
    REGT_CUDA(cudaMemsetAsync(rseg_ptr, 0, sizeof(int32_t) * (R + 1), st));
    REGT_CUDA(cudaMemsetAsync(seg_ptr, 0, sizeof(int32_t) * (N + 1), st));
    REGT_CUDA(cudaMemsetAsync(seg_eptr, 0, sizeof(int32_t), st));
  }
  REGT_CUDA(cudaStreamSynchronize(st));
  if (counts_out) {
    counts_out[0] = nnz;
    counts_out[1] = nseg;
  }
  return 0;
}
