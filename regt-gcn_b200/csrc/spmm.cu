// F-wide CSR SpMM over the x[B,N,F,T] layout of the reference (load_dataset.py:456).
//
// Because T is the innermost dimension of x, one neighbour row x[b,j,:,:] is F*T
// contiguous floats (96 floats = 384 B at T=12): a single gather serves all T periods,
// so  S[b,n,:,:] = sum_e A_hat[e] * x[b,col[e],:,:]  is one SpMM on 384-byte rows instead
// of 3*T scatter-add passes on 1 KB rows (GCNConv.propagate, models/utils.py:169,175,181).
// HBM-bound: algorithmic bytes = read x once + write y once + CSR (SURVEY 8(d) SpMMBytes).
//
// One warp per output row; lane c owns float4 #c of the row (128-bit loads/stores, fully
// coalesced 384 B per neighbour); edge metadata is read once per warp (uniform address).
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace regt {

__device__ __forceinline__ float4 ld_nc4(const float4* p) { return __ldg(p); }

template <int UNROLL>
__global__ void __launch_bounds__(256) k_spmm_rows(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                   const float* __restrict__ val, const float4* __restrict__ x,
                                                   float4* __restrict__ y, int B, int n_out, int n_in, int W4) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (warp >= (long long)B * n_out) return;
  const int b = (int)(warp / n_out), r = (int)(warp % n_out);
  const float4* xb = x + (size_t)b * n_in * W4;
  float4* yr = y + ((size_t)b * n_out + r) * W4;
  const int e0 = rowptr[r], e1 = rowptr[r + 1];
  for (int c = lane; c < W4; c += 32) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int e = e0;
    for (; e + UNROLL <= e1; e += UNROLL) {
      float4 v[UNROLL];
      float w[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        w[u] = __ldg(val + e + u);
        v[u] = ld_nc4(xb + (size_t)__ldg(col + e + u) * W4 + c);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {  // sequential CSR order: deterministic sums
        acc.x = fmaf(w[u], v[u].x, acc.x);
        acc.y = fmaf(w[u], v[u].y, acc.y);
        acc.z = fmaf(w[u], v[u].z, acc.z);
        acc.w = fmaf(w[u], v[u].w, acc.w);
      }
    }
    for (; e < e1; ++e) {
      float w = __ldg(val + e);
      float4 v = ld_nc4(xb + (size_t)__ldg(col + e) * W4 + c);
      acc.x = fmaf(w, v.x, acc.x);
      acc.y = fmaf(w, v.y, acc.y);
      acc.z = fmaf(w, v.z, acc.z);
      acc.w = fmaf(w, v.w, acc.w);
    }
    yr[c] = acc;
  }
}

// Shared-memory staged variant (north_star: "warp-per-row CSR gather ... shared-memory staging of neighbour feature
// tiles").  A block of NB consecutive nodes of one snapshot is ONE contiguous run of NB * W floats in x[b]: it is pulled
// into shared memory with the bulk-copy engine (DRAM -> smem, no register round trip), then the block's rows are
// gathered from shared memory whenever the neighbour lies in the block (road graphs: regions are contiguous id ranges, so
// most neighbours do) and from global memory (L2) otherwise.  The warp-per-row kernel above reads every neighbour row
// through L2 -- 7.1 x 384 B per output row at config 5 against 768 B of DRAM traffic -- and runs L2-gather-bound; here
// the L2 side shrinks to the block load plus the out-of-block neighbours.  Same sequential CSR order and the same fmaf
// chain as k_spmm_rows: bit-identical results.
// v2 (this round): the block's CSR slice (rowptr, col, val -- contiguous, because the rows are) is staged too, so the
// edge loop has no dependent global loads (v1 read col/val per edge through L2: 2.67 ms at config 5, latency-bound, 0.28
// of the HBM peak), and two CTAs share an SM so that one's block load overlaps the other's gather.
constexpr int SPMM_EDGES_PER_SM = 3584;  // staged edges per SM, split between its resident CTAs (more: the tail is read from global memory)
// v3: the kernel was ISSUE-bound (ncu: 70 % issue-active, integer compares and address arithmetic around four FMAs per
// edge and lane).  The staging threads resolve every edge ONCE per block.
// v4: ... into the GENERIC address of the neighbour row -- inside the staged block (shared window) or in x (global) --
// plus the weight, one 16-byte word.  ncu of v3 counted 290 warp instructions per output row (about 30 per edge: both
// sides of the staged / not-staged choice are predicated, not branched, so each costs issue slots); with one address space
// the gather loop is a broadcast LDS.128, a 64-bit add, one generic 128-bit load and four FMAs.
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
struct __align__(16) SpmmEdge {
  const float4* row;     // generic pointer: staged copy of the neighbour row, or the row in global memory
  float w;
  int pad;
};
template <int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_spmm_blk(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                                  const float* __restrict__ val, const float4* __restrict__ x,
                                                                  float4* __restrict__ y, int B, int n_out, int n_in, int W4, int NB,
                                                                  int nblk, const int32_t* __restrict__ blk_ptr) {
  constexpr int SPMM_EMAX = SPMM_EDGES_PER_SM / MINB;
  extern __shared__ __align__(128) uint8_t spmm_smem[];
  __shared__ uint64_t bar;
  float4* xs = reinterpret_cast<float4*>(spmm_smem);
  int32_t* s_ptr = reinterpret_cast<int32_t*>(spmm_smem + (size_t)NB * W4 * 16);   // [NB + 1] edge offsets relative to the block's first edge
  SpmmEdge* s_edge = reinterpret_cast<SpmmEdge*>(s_ptr + ((NB + 1 + 3) & ~3));     // [SPMM_EMAX]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  if (threadIdx.x == 0) {
    tc::mbar_init(&bar, 1);
    tc::fence_barrier_init();
  }
  __syncthreads();
  uint32_t phase = 0;
  // The CSR slice of an item (row offsets, neighbour ids, weights) is fetched into REGISTERS one item ahead: its two
  // dependent L2 round trips (rowptr -> col / val) then run under the bulk load of the current block instead of in front of it.
  constexpr int PER = (SPMM_EMAX + NT - 1) / NT;
  struct Meta {
    int r0, r1, s1, eb, ne, sp;
    int jj[PER];
    float ww[PER];
  };
  const long long n_items = (long long)B * nblk;
  auto fetch = [&](long long item, Meta& m) {
    const int blk = (int)(item % nblk);
    // uniform blocks of NB rows, or the plan's partition (regt_spmm_partition: row ranges of at most NB rows, cut where
    // the fewest edges cross, so that nearly every neighbour of a block lies inside it)
    m.r0 = blk_ptr ? __ldg(blk_ptr + blk) : blk * NB;
    m.r1 = blk_ptr ? __ldg(blk_ptr + blk + 1) : min(n_out, m.r0 + NB);
    m.s1 = blk_ptr ? m.r1 : min(n_in, m.r0 + NB);        // staged node range [r0, s1)
    m.eb = __ldg(rowptr + m.r0);
    const int ee = __ldg(rowptr + m.r1);
    m.sp = ((int)threadIdx.x <= m.r1 - m.r0) ? __ldg(rowptr + m.r0 + threadIdx.x) : 0;
    m.ne = min(ee - m.eb, SPMM_EMAX);
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int i = threadIdx.x + u * NT;
      m.jj[u] = 0;
      m.ww[u] = 0.f;
      if (i < m.ne) {
        m.jj[u] = __ldg(col + m.eb + i);
        m.ww[u] = __ldg(val + m.eb + i);
      }
    }
  };
  Meta cur;
  if ((long long)blockIdx.x < n_items) fetch(blockIdx.x, cur);
  for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    // items are ordered snapshot-major: the CTAs running side by side work on neighbouring node blocks of ONE snapshot, so
    // an out-of-block neighbour row is (still) in L2 because the CTA next door staged it
    const int b = (int)(item / nblk);
    const int r0 = cur.r0, r1 = cur.r1, s1 = cur.s1, eb = cur.eb;
    const float4* xb = x + (size_t)b * n_in * W4;
    const long long nxt = item + gridDim.x;
    if (threadIdx.x == 0) {
      const uint32_t bytes = (uint32_t)(s1 - r0) * W4 * 16;
      tc::mbar_arrive_expect_tx(&bar, bytes);
      const uint8_t* src = reinterpret_cast<const uint8_t*>(xb + (size_t)r0 * W4);
      for (uint32_t o = 0; o < bytes; o += 32768) tc::bulk_g2s(spmm_smem + o, src + o, min(32768u, bytes - o), &bar);
      // the NEXT item's rows start their way from DRAM into L2 now: with one CTA per SM nothing overlaps the block load, so
      // it should at least be an L2 read
      if (nxt < n_items) {
        const int nb2 = (int)(nxt / nblk), k2 = (int)(nxt - (long long)nb2 * nblk);
        const int q0 = blk_ptr ? __ldg(blk_ptr + k2) : k2 * NB;
        const int q1 = blk_ptr ? __ldg(blk_ptr + k2 + 1) : min(n_in, q0 + NB);
        const uint8_t* s2 = reinterpret_cast<const uint8_t*>(x + ((size_t)nb2 * n_in + q0) * W4);
        const uint32_t by2 = (uint32_t)(q1 - q0) * W4 * 16;
        for (uint32_t o = 0; o < by2; o += 32768) tc::bulk_prefetch_l2(s2 + o, min(32768u, by2 - o));
      }
    }
    // this item's slice: registers -> shared memory, every edge resolved to the generic address of its neighbour row
    if ((int)threadIdx.x <= r1 - r0) s_ptr[threadIdx.x] = cur.sp - eb;
    if (NT <= NB)
      for (int i = threadIdx.x + NT; i <= r1 - r0; i += NT) s_ptr[i] = __ldg(rowptr + r0 + i) - eb;   // blocks of more rows than threads
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int i = threadIdx.x + u * NT;
      if (i < cur.ne) {
        const int j = cur.jj[u];
        SpmmEdge ed;
        ed.row = (j >= r0 && j < s1) ? xs + (size_t)(j - r0) * W4 : xb + (size_t)j * W4;
        ed.w = cur.ww[u];
        ed.pad = 0;
        s_edge[i] = ed;
      }
    }
    if (nxt < n_items) fetch(nxt, cur);
    __syncthreads();
    tc::mbar_wait(&bar, phase);
    phase ^= 1;
    // One 16-byte broadcast load per edge (inline asm: field-wise the struct read becomes LDS.64 + LDS.32), two edges per
    // trip and an odd one after the loop -- at ~7 edges per row a deeper unroll spends more on its remainder tree than it
    // saves (ncu, v4 first cut: 181 warp instructions per row, a third of them loop control).
    const uint32_t s_e4 = tc::smem_u32(s_edge);
    float4* yb = y + ((size_t)b * n_out + r0) * W4;
    const int nrows = r1 - r0;
    for (int c = lane; c < W4; c += 32) {       // one pass for rows of up to 32 float4 (F*T = 96 floats: 24 lanes)
      for (int rr = warp; rr < nrows; rr += nwarp) {
        const int e0 = s_ptr[rr], e1 = s_ptr[rr + 1];
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t ea = s_e4 + (uint32_t)e0 * 16u;
        const uint32_t ee4 = s_e4 + (uint32_t)min(e1, SPMM_EMAX) * 16u;
        // (Loading the entries of the next trip before this trip's rows are used -- one shared-memory round trip on the
        // critical path instead of two -- measured slower, 3.20 against 3.36 TB/s: the gather is bound by shared-memory
        // wavefronts, 5 per edge (2 for the broadcast entry, 3 for the 384-byte row), not by the latency of the chain.)
#pragma unroll 1
        for (; ea + 32u <= ee4; ea += 32u) {        // sequential CSR order: deterministic sums
          const uint4 q0 = lds128(ea), q1 = lds128(ea + 16u);
          const float4 v0 = reinterpret_cast<const float4*>(((unsigned long long)q0.y << 32) | q0.x)[c];
          const float4 v1 = reinterpret_cast<const float4*>(((unsigned long long)q1.y << 32) | q1.x)[c];
          const float w0 = __uint_as_float(q0.z), w1 = __uint_as_float(q1.z);
          acc.x = fmaf(w0, v0.x, acc.x);
          acc.y = fmaf(w0, v0.y, acc.y);
          acc.z = fmaf(w0, v0.z, acc.z);
          acc.w = fmaf(w0, v0.w, acc.w);
          acc.x = fmaf(w1, v1.x, acc.x);
          acc.y = fmaf(w1, v1.y, acc.y);
          acc.z = fmaf(w1, v1.z, acc.z);
          acc.w = fmaf(w1, v1.w, acc.w);
        }
        if (ea < ee4) {
          const uint4 q0 = lds128(ea);
          const float4 v0 = reinterpret_cast<const float4*>(((unsigned long long)q0.y << 32) | q0.x)[c];
          const float w0 = __uint_as_float(q0.z);
          acc.x = fmaf(w0, v0.x, acc.x);
          acc.y = fmaf(w0, v0.y, acc.y);
          acc.z = fmaf(w0, v0.z, acc.z);
          acc.w = fmaf(w0, v0.w, acc.w);
        }
        if (e1 > SPMM_EMAX) {                 // edges beyond the staged slice (blocks with very many edges)
          for (int e = max(e0, SPMM_EMAX); e < e1; ++e) {
            const int j = __ldg(col + eb + e);
            const float w = __ldg(val + eb + e);
            const float4 v = (j >= r0 && j < s1) ? xs[(size_t)(j - r0) * W4 + c] : __ldg(xb + (size_t)j * W4 + c);
            acc.x = fmaf(w, v.x, acc.x);
            acc.y = fmaf(w, v.y, acc.y);
            acc.z = fmaf(w, v.z, acc.z);
            acc.w = fmaf(w, v.w, acc.w);
          }
        }
        yb[(unsigned)(rr * W4 + c)] = acc;
      }
    }
    __syncthreads();     // every warp is done with the staged block before the next one lands
  }
}

// Feature builder of the tensor-core path: the results are written period-major so that one (tile, period) of the
// cell kernels reads contiguous 32-byte rows:
//   Xt[t][q][F] = x[q][:, t]      St[t][q][F] = (A_hat x)[q][:, t]      Ut[t][b*nseg+s][F] = (L_hat_r x) per segment
// One THREAD per (row, period), period fastest: the 12 period-threads of a row read a neighbour's whole 384-byte
// feature row between them (48-byte runs per feature), the edge metadata of a row is a broadcast load, and each
// thread writes its own 32-byte output row -- no shuffles, no staging, ~4x fewer instructions than the warp-per-row
// gather (which spent its time on issue slots and three dependent memory rounds at 37 % occupancy).  Sums stay in
// sequential CSR order (bit-identical to the stand-alone SpMM).  x has FIN <= F features per node (row stride FIN*T): only
// those are gathered, the output rows stay F wide with zeros in FIN..F-1.
#ifndef REGT_FEAT_MINB
#define REGT_FEAT_MINB 4
#endif
template <int FIN>
__global__ void __launch_bounds__(256, REGT_FEAT_MINB) k_feat_tc(const int32_t* __restrict__ g_rowptr, const int32_t* __restrict__ g_col,
                                                 const float* __restrict__ g_val, const int32_t* __restrict__ seg_eptr,
                                                 const int32_t* __restrict__ c_col, const float* __restrict__ c_val,
                                                 const float* __restrict__ x, int B, int N, int xN, int nseg, int T,
                                                 float* __restrict__ Xt, float* __restrict__ St, float* __restrict__ Ut) {
  constexpr int F = REGT_F;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long BN = (long long)B * N, BS = (long long)B * nseg;
  const long long nA = BN * T;
  if (i >= nA + BS * T) return;
  const bool is_seg = i >= nA;
  const long long j = is_seg ? i - nA : i;
  const long long w = j / T;                       // b * N + r   (or b * nseg + s)
  const int t = (int)(j - w * T);
  const int per = is_seg ? nseg : N;
  const int b = (int)(w / per), r = (int)(w - (long long)b * per);
  const int* rowptr = is_seg ? seg_eptr : g_rowptr;
  const int* col = is_seg ? c_col : g_col;
  const float* val = is_seg ? c_val : g_val;
  const int W = FIN * T;
  const float* xb = x + (size_t)b * xN * W + t;    // element (node, f) of this sample and period: xb[node * W + f * T]
  const int e0 = __ldg(rowptr + r), e1 = __ldg(rowptr + r + 1);
  float acc[F];
#pragma unroll
  for (int f = 0; f < F; ++f) acc[f] = 0.f;       // features FIN.. stay zero
  int e = e0;
  for (; e + 4 <= e1; e += 4) {   // four edges' loads in flight, accumulated in CSR order
    int c4[4];
    float v4[4], xv[4][FIN];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      c4[u] = __ldg(col + e + u);
      v4[u] = __ldg(val + e + u);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float* xr = xb + (size_t)c4[u] * W;
#pragma unroll
      for (int f = 0; f < FIN; ++f) xv[u][f] = __ldg(xr + f * T);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int f = 0; f < FIN; ++f) acc[f] = fmaf(v4[u], xv[u][f], acc[f]);
  }
  for (; e < e1; ++e) {
    const float v = __ldg(val + e);
    const float* xr = xb + (size_t)__ldg(col + e) * W;
#pragma unroll
    for (int f = 0; f < FIN; ++f) acc[f] = fmaf(v, __ldg(xr + f * T), acc[f]);
  }
  float4* d = reinterpret_cast<float4*>((is_seg ? Ut : St) + ((size_t)t * (is_seg ? BS : BN) + w) * F);
  d[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
  d[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  if (!is_seg) {
    const float* xr = xb + (size_t)r * W;
    float sx[F];
#pragma unroll
    for (int f = 0; f < F; ++f) sx[f] = f < FIN ? __ldg(xr + f * T) : 0.f;
    float4* dx = reinterpret_cast<float4*>(Xt + ((size_t)t * BN + w) * F);
    dx[0] = make_float4(sx[0], sx[1], sx[2], sx[3]);
    dx[1] = make_float4(sx[4], sx[5], sx[6], sx[7]);
  }
}

int launch_feat_tc(const regt_graph_plan& p, const float* x, int Fin, int B, int xN, int T, float* Xt, float* St, float* Ut,
                   cudaStream_t st) {
  const long long threads = ((long long)B * p.N + (long long)B * p.nseg) * T;
  auto kern = k_feat_tc<8>;
  switch (Fin) {
    case 1: kern = k_feat_tc<1>; break;
    case 2: kern = k_feat_tc<2>; break;
    case 3: kern = k_feat_tc<3>; break;
    case 4: kern = k_feat_tc<4>; break;
    case 5: kern = k_feat_tc<5>; break;
    case 6: kern = k_feat_tc<6>; break;
    case 7: kern = k_feat_tc<7>; break;
    case 8: break;
    default: REGT_CHECK(false, "feat_tc: %d node features, the kernels take 1..%d", Fin, REGT_F);
  }
  kern<<<cdiv(threads, 256), 256, 0, st>>>(p.g_rowptr, p.g_col, p.g_val, p.seg_eptr, p.c_col, p.c_val, x, B, p.N, xN, p.nseg, T, Xt, St,
                                           Ut);
  REGT_LAUNCHED("k_feat_tc", st);
  return 0;
}

// xw[q][f][t] = f < Fin ? x[q][f][t] : 0 for every row q of x (halo rows included): the FFMA and unfused tf32x3 kernels
// read x through several launches at REGT_F features per row.  Scalar loads: x needs 4-byte alignment only.
__global__ void k_widen_x(const float* __restrict__ x, int Fin, int T, long long total, float* __restrict__ xw) {
  constexpr int F = REGT_F;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long q = i / ((long long)F * T);
  const int rem = (int)(i - q * F * T), f = rem / T, t = rem - f * T;
  xw[i] = f < Fin ? __ldg(x + (q * Fin + f) * T + t) : 0.f;
}

int launch_widen_x(const regt_args* a, const Layout& L, cudaStream_t st) {
  if (!L.xw) return 0;
  const long long total = (long long)a->B * (a->x_rows > 0 ? a->x_rows : a->N) * REGT_F * a->T;
  k_widen_x<<<cdiv(total, 256), 256, 0, st>>>(a->x, feat_in(a), a->T, total, L.xw);
  REGT_LAUNCHED("k_widen_x", st);
  return 0;
}

// staged-kernel geometry for rows of `width` floats: row capacity of a block, staged edges.  One 1024-thread CTA per SM with
// the whole shared memory measured fastest on config 5 (3.07 TB/s against 2.67 with two CTAs of half the rows: the larger
// block keeps more neighbours staged, which matters more than overlapping one CTA's block load with the other's gather).
static inline void spmm_geometry(int width, int* nb_cap, int* emax) {
  *emax = SPMM_EDGES_PER_SM;
  *nb_cap = (227 * 1024 - 2048 - *emax * 16 - 64) / (width * 4 + 4) / 8 * 8;
}

int launch_spmm_impl(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y, int B,
                     int n_out, int n_in, int width, const int32_t* blk_ptr, int nblk_p, cudaStream_t st) {
  REGT_CHECK(width % 4 == 0 && width > 0, "spmm: width %d must be a positive multiple of 4", width);
  if (B == 0 || n_out == 0) return 0;
  // staged variant: output row r <-> node r (square operator, possibly with halo columns behind the rows), blocks of
  // NB nodes = up to 192 KB of shared memory; small problems keep the plain warp-per-row kernel (less than one wave)
  const int row_bytes = width * 4;
  int emax, NB;
  spmm_geometry(width, &NB, &emax);
  REGT_CHECK(!blk_ptr || (NB >= 32 && n_out == n_in && nblk_p > 0 && ((uintptr_t)x % 16) == 0),
             "spmm: a partition needs a square operator, 16-byte aligned x and rows that fit the staged kernel (width %d)", width);
  if (blk_ptr || (n_out <= n_in && NB >= 32 && (long long)B * n_out >= 4096 && ((uintptr_t)x % 16) == 0)) {
    int nblk = nblk_p;
    if (!blk_ptr) {
      NB = min(NB, (n_out + 7) / 8 * 8);
      // balance the blocks of a snapshot (a short last block would idle an SM for most of a wave)
      nblk = cdiv(n_out, NB);
      NB = (cdiv(n_out, nblk) + 7) / 8 * 8;
    }
    const size_t smem = (size_t)NB * row_bytes + (size_t)((NB + 1 + 3) & ~3) * 4 + (size_t)emax * 16;
    static int sms = 0;
    if (sms == 0) {
      int dev = 0;
      if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    const long long items = (long long)B * nblk;
    const int grid = (int)min(items, (long long)sms);
    REGT_CUDA(cudaFuncSetAttribute(k_spmm_blk<1024, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_spmm_blk<1024, 1><<<grid, 1024, smem, st>>>(rowptr, col, val, (const float4*)x, (float4*)y, B, n_out, n_in, width / 4, NB, nblk, blk_ptr);
    REGT_LAUNCHED("k_spmm_blk", st);
    return 0;
  }
  long long warps = (long long)B * n_out;
  k_spmm_rows<4><<<cdiv(warps * 32, 256), 256, 0, st>>>(rowptr, col, val, (const float4*)x, (float4*)y, B, n_out, n_in,
                                                       width / 4);
  REGT_LAUNCHED("k_spmm_rows", st);
  return 0;
}
int launch_spmm_rows(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y, int B,
                     int n_out, int n_in, int width, cudaStream_t st) {
  return launch_spmm_impl(rowptr, col, val, x, y, B, n_out, n_in, width, nullptr, 0, st);
}

// Plan-time partition of the rows into the staged kernel's blocks (host side: the CSR is copied back once per static graph,
// like the counts of the *_plan_build calls).  span[p] = number of edges (i, j) with min(i, j) < p <= max(i, j), i.e. the
// neighbour reads that leave their block if a block boundary is put in front of row p; boundaries are chosen greedily in the
// upper half of each block's admissible window, at the smallest span (ties: the longest block).  On graphs whose node ids
// are ordered by region (the reference's regional edge lists are contiguous id ranges) the cuts fall on the region borders.
static int spmm_partition_host(const std::vector<int32_t>& rp, const std::vector<int32_t>& cj, int N, int nb_cap, int emax,
                               std::vector<int32_t>* out) {
  std::vector<int32_t> span((size_t)N + 2, 0);
  for (int i = 0; i < N; ++i)
    for (int e = rp[i]; e < rp[i + 1]; ++e) {
      const int j = cj[e];
      if (j < 0 || j >= N || j == i) continue;
      const int lo = i < j ? i : j, hi = i < j ? j : i;
      span[lo + 1] += 1;
      span[hi + 1] -= 1;
    }
  for (int p = 1; p <= N; ++p) span[p] += span[p - 1];
  out->clear();
  out->push_back(0);
  int s0 = 0;
  while (s0 < N) {
    int lim = s0 + 1;                                   // the furthest admissible end: rows and staged edges both fit
    while (lim < N && lim + 1 - s0 <= nb_cap && rp[lim + 1] - rp[s0] <= emax) ++lim;
    int cut = lim;
    if (lim < N) {
      const int lo = s0 + (lim - s0 + 1) / 2;
      for (int p = lim; p >= lo && p > s0; --p)
        if (span[p] < span[cut]) cut = p;
    }
    out->push_back(cut);
    s0 = cut;
  }
  return (int)out->size() - 1;
}

// K4 regional gather / scatter of node rows (region shards: owned + halo rows in, owned rows out)
//   gather : dst[b][i][:] = src[b][idx[i]][:]   i < n_idx   (src has n_src rows, dst n_idx rows)
//   scatter: dst[b][idx[i]][:] = src[b][i][:]   i < n_idx   (src has n_idx rows, dst n_dst rows)
template <bool SCATTER, typename V>
__global__ void __launch_bounds__(256) k_move_rows(const V* __restrict__ src, const int64_t* __restrict__ idx,
                                                   V* __restrict__ dst, int n_idx, int n_other, int WV, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % WV);
  const long long br = i / WV;
  const int r = (int)(br % n_idx), b = (int)(br / n_idx);
  const size_t packed = ((size_t)b * n_idx + r) * WV + c;
  const size_t strided = ((size_t)b * n_other + (size_t)__ldg(idx + r)) * WV + c;
  if (SCATTER) dst[strided] = src[packed];
  else dst[packed] = __ldg(src + strided);
}

template <bool SCATTER>
static int launch_move_rows(const float* src, const int64_t* idx, float* dst, int B, int n_idx, int n_other, int width,
                            cudaStream_t st) {
  REGT_CHECK(src && idx && dst, "gather/scatter_rows: NULL pointer");
  REGT_CHECK(B >= 0 && n_idx >= 0 && n_other >= 0 && width > 0, "gather/scatter_rows: bad sizes");
  if (B == 0 || n_idx == 0) return 0;
  const bool v4 = width % 4 == 0 && ((uintptr_t)src % 16 == 0) && ((uintptr_t)dst % 16 == 0);
  const int WV = v4 ? width / 4 : width;
  const long long total = (long long)B * n_idx * WV;
  if (v4) k_move_rows<SCATTER, float4><<<cdiv(total, 256), 256, 0, st>>>((const float4*)src, idx, (float4*)dst, n_idx, n_other, WV, total);
  else k_move_rows<SCATTER, float><<<cdiv(total, 256), 256, 0, st>>>(src, idx, dst, n_idx, n_other, WV, total);
  REGT_LAUNCHED(SCATTER ? "k_scatter_rows" : "k_gather_rows", st);
  return 0;
}

}  // namespace regt

extern "C" int regt_gather_rows(const float* src, const int64_t* idx, float* dst, int32_t B, int32_t n_src, int32_t n_idx,
                                int32_t width, regt_stream_t stream) {
  return regt::launch_move_rows<false>(src, idx, dst, B, n_idx, n_src, width, (cudaStream_t)stream);
}
extern "C" int regt_scatter_rows(const float* src, const int64_t* idx, float* dst, int32_t B, int32_t n_idx, int32_t n_dst,
                                 int32_t width, regt_stream_t stream) {
  return regt::launch_move_rows<true>(src, idx, dst, B, n_idx, n_dst, width, (cudaStream_t)stream);
}

extern "C" int32_t regt_spmm_partition_capacity(int32_t N, int32_t width) {
  if (N <= 0 || width <= 0 || width % 4) return 0;
  int nb, emax;
  regt::spmm_geometry(width, &nb, &emax);
  if (nb < 32) return 0;                                // rows too wide for the staged kernel: no partition
  return N + 2;                                         // worst case: one block per row (rows with more edges than a block stages)
}
extern "C" int regt_spmm_partition(const int32_t* rowptr, const int32_t* col, int32_t N, int32_t width, int32_t* blk_ptr,
                                   int32_t* nblk_out, regt_stream_t stream) {
  REGT_CHECK(rowptr && col && blk_ptr && nblk_out, "spmm_partition: NULL pointer");
  REGT_CHECK(regt_spmm_partition_capacity(N, width) > 0, "spmm_partition: N %d / width %d not supported by the staged kernel", N, width);
  cudaStream_t st = (cudaStream_t)stream;
  int nb, emax;
  regt::spmm_geometry(width, &nb, &emax);
  std::vector<int32_t> rp((size_t)N + 1);
  REGT_CUDA(cudaMemcpyAsync(rp.data(), rowptr, sizeof(int32_t) * ((size_t)N + 1), cudaMemcpyDeviceToHost, st));
  REGT_CUDA(cudaStreamSynchronize(st));
  REGT_CHECK(rp[0] == 0 && rp[N] >= 0, "spmm_partition: bad rowptr");
  std::vector<int32_t> cj((size_t)rp[N]);
  if (rp[N]) REGT_CUDA(cudaMemcpyAsync(cj.data(), col, sizeof(int32_t) * (size_t)rp[N], cudaMemcpyDeviceToHost, st));
  REGT_CUDA(cudaStreamSynchronize(st));
  std::vector<int32_t> blk;
  const int nblk = regt::spmm_partition_host(rp, cj, N, nb, emax, &blk);
  REGT_CUDA(cudaMemcpyAsync(blk_ptr, blk.data(), sizeof(int32_t) * blk.size(), cudaMemcpyHostToDevice, st));
  REGT_CUDA(cudaStreamSynchronize(st));
  *nblk_out = nblk;
  return 0;
}
// TEST HOOK: the partition algorithm on HOST arrays (no device work): what regt_spmm_partition computes after copying the CSR back
extern "C" int regt_debug_spmm_partition_host(const int32_t* rowptr, const int32_t* col, int32_t N, int32_t width, int32_t* blk_ptr,
                                              int32_t* nblk_out, int32_t* cap_out) {
  REGT_CHECK(rowptr && col && blk_ptr && nblk_out && N > 0 && width > 0 && width % 4 == 0, "spmm_partition_host: bad arguments");
  int nb, emax;
  regt::spmm_geometry(width, &nb, &emax);
  REGT_CHECK(nb >= 32, "spmm_partition_host: rows of %d floats do not fit the staged kernel", width);
  std::vector<int32_t> rp(rowptr, rowptr + N + 1), cj(col, col + rowptr[N]), blk;
  *nblk_out = regt::spmm_partition_host(rp, cj, N, nb, emax, &blk);
  for (size_t i = 0; i < blk.size(); ++i) blk_ptr[i] = blk[i];
  if (cap_out) { cap_out[0] = nb; cap_out[1] = emax; }
  return 0;
}
extern "C" int regt_spmm_f8_blocked(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y,
                                    int32_t B, int32_t N, int32_t width, const int32_t* blk_ptr, int32_t nblk,
                                    regt_stream_t stream) {
  REGT_CHECK(blk_ptr && nblk > 0, "spmm_f8_blocked: no partition (regt_spmm_partition)");
  return regt::launch_spmm_impl(rowptr, col, val, x, y, B, N, N, width, blk_ptr, nblk, (cudaStream_t)stream);
}

extern "C" int regt_spmm_f8(const int32_t* rowptr, const int32_t* col, const float* val, const float* x, float* y,
                            int32_t B, int32_t N, int32_t width, regt_stream_t stream) {
  return regt::launch_spmm_rows(rowptr, col, val, x, y, B, N, N, width, (cudaStream_t)stream);
}
