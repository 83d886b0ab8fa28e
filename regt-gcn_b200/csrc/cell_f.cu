// Fused fp32-parity (3xTF32) cell for hidden = 128 / 64: the tensor-core gate GEMMs, the GRU nonlinearities, the
// period-attention sum and their backward data gradients in TWO persistent kernels (one CTA per SM), instead of the
// five GEMM launches + seven elementwise passes of cell_g.cu.  Per (b,n,t) row the forward writes three H-wide planes
// (Z, R, H~) and nothing else; the unfused path moves ~17 plane passes forward and ~27 backward.
//
// What makes H = 128 fit (cell_tc.cu's design needs the weights resident in shared memory: 442 KB here):
//   * the A operand (h, then h*R; the gate gradients in the backward) lives in TENSOR MEMORY as tf32 hi | lo column
//     blocks -- written by the epilogue threads with tcgen05.st, read by "TS" MMAs -- so shared memory holds no A tile;
//   * the split weights stream from L2 through a ring of 32 KB stages ([128 n][32 k] hi | lo, SW128 K-major, already in
//     UMMA layout in a per-step global image): a producer thread cycles the same 12 stages per (tile, period) with the
//     bulk-copy engine and runs ahead of the MMAs by the depth of the ring, across tile boundaries;
//   * TMEM = 512 columns exactly: A hi | A lo (2H) + two H-wide accumulators that are re-used within a step
//     (forward: z | r, then the candidate in r's columns; backward: dHR | dhg).
//
// Work item = 128 rows (b,n) x ALL T periods: thread (row, H/2 columns) keeps  sum_t probs[t] H'_t  in registers.
//
// Forward step (tile, t):            P   h = act(X_t M0 + U_t M1[r] + c0) on the CUDA cores -> TMEM A (hi | lo); S_t tile -> smem
//   MMA z : acc_z = [h | S] Wz       E1z Z = sigmoid(.), save Z, acc += p Z h                 (under MMA r)
//   MMA r : acc_r = [h | S] Wr       E1r R = sigmoid(.), save R, h*R -> TMEM A
//   MMA c : acc_c = [h*R | S] Wc     P(next step) as soon as MMA c is done -> MMA z(next) starts, then
//                                    E2  H~ = tanh(.), save H~, acc += p (1 - Z) H~          (under MMA z of the next step)
// Backward step: E0 recompute h, read Z,R,H~,G -> Dc (TMEM A), Dz (registers), planes h, h*R, Dz, Dc, d probs
//   M1 dHR = Dc B_h ; Dz -> A ; M2z dhg = Dz B_z (E1 under it: Dr = dHR h R(1-R), t1 = dHR R kept in TMEM) ; Dr -> A ;
//   M2r dhg += Dr B_r ; E2 d h_pre = act'(h)(p G Z + t1 + dhg).  The four gate-gradient blocks D, h and h*R go to HBM row
//   major (row = t * BNp + q) for the weight-gradient row contraction (gemm_tma.cu), which cannot live here: its
//   accumulators alone (3 H x H + 4H x 32 fp32) exceed TMEM.
// Reference arithmetic replaced: models/utils.py:168-188, models/RegionalTemporalGCN.py:134-148, models/TemporalGCN.py:84-90.
#include <stdlib.h>

#include "cell_tc.cuh"

namespace regt {
using namespace tc;

// phase timestamps of CTA 0 / epilogue thread 0 (REGT_F_DEBUG=1; read back with regt_debug_f_timestamps): 16 steps x 12 marks
__device__ long long g_f_dbg[3][16 * 12];      // [2]: marks of the forward's MMA warp (lane 0)
#define F_TSM(i)                                                                              \
  if (a.dbg && blockIdx.x == 0 && lane == 0 && s >= a.dbg && s < a.dbg + 16) g_f_dbg[2][(s - a.dbg) * 12 + (i)] = clock64();
#define F_TS(which, i)                                                                        \
  if (a.dbg && blockIdx.x == 0 && tid == 0 && s >= a.dbg && s < a.dbg + 16) g_f_dbg[which][(s - a.dbg) * 12 + (i)] = clock64();

namespace {
constexpr int F = REGT_F;
// 16 epilogue warps = 4 TMEM lane quarters x 4 column groups.  With 8 warps (two per scheduler) the epilogue phases were
// latency-bound chains -- ncu: 50-60 % of the samples on long-scoreboard stalls, tensor pipe 24 % busy forward / 13 % backward
// (profiles/r02_cell_f_v1_ncu.md) -- so the thread count doubled (4 warps per scheduler, half the columns per thread).
constexpr int NEPI_W = 16;
// Register split (setmaxnreg): the launch gives every warp the same count -- 96 at 640 threads (5 warps per scheduler
// partition x 96 x 32 <= 16 K registers) -- which spills in the epilogue threads.  The fifth warpgroup (MMA issuer, weight
// producer, two idle warps) drops to REGS_AUX and each epilogue warp grows to REGS_EPI: the pool is per CTA: 16 warps x (112 - 96) = 4 warps x (96 - 32).
constexpr int REGS_EPI = 112, REGS_AUX = 32;
__device__ __forceinline__ void regs_grow() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI)); }
__device__ __forceinline__ void regs_shrink() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_AUX)); }
constexpr int W_MMA = NEPI_W;             // issues every tcgen05.mma (one elected lane), owns the TMEM allocation
constexpr int W_PROD = NEPI_W + 1;        // weight-stage producer (bulk copies); warps NEPI_W + 2, + 3 only complete the warpgroup
constexpr int NTHR = (NEPI_W + 4) * 32;
constexpr int SMEM_MAX = 227 * 1024;

template <int HH>
struct FCfg {
  static constexpr int NCH = HH / 32;                 // K chunks (32 tf32 = one 128-byte swizzle row) of an H-wide block
  static constexpr int TILE = HH * 128;               // [HH n][32 k] tf32, SW128 K-major
  static constexpr int STAGE = 2 * TILE;              // hi | lo
  static constexpr int NSTEP = 3 * NCH;               // stages consumed per (tile, period): three H x H blocks
  static constexpr int RING_IMG = NSTEP * STAGE;
  static constexpr int SW_TILE = 2 * HH * 16;         // F-wide (S) part of one gate: chunk tile [2 chunks][HH n][16 B]
  static constexpr int SW_IMG = 3 * 2 * SW_TILE;      // 3 gates x (hi | lo)
  static constexpr int C_CZR = 0, C_CC = 2 * HH, C_C0 = 3 * HH, C_M0 = 4 * HH, C_M1 = 12 * HH, C_PROBS = 20 * HH,
                       C_FLOATS = 20 * HH + 64;
  static constexpr int TAIL = SW_IMG + C_FLOATS * 4;  // resident part of the image (copied once per CTA)
  static constexpr int IMG = RING_IMG + TAIL;
  static constexpr int S_TILE = 2 * TC_ROWS * 16;     // A operand of the F-wide part: S_t (8 tf32) per row, chunk tile
  // h_pre on the tensor cores (forward, regional mode): A = [X | U.1(r = ra) | U.1(r = rb)] per row, three K = 8 chunk tiles
  // (hi | lo), B = [M0 ; M1[ra] ; M1[rb]]^T of the item, three chunk tiles (hi | lo)
  static constexpr int XU_TILE = 3 * 2 * S_TILE;
  static constexpr int WP_TILE = 3 * 2 * SW_TILE;
  static constexpr int FIXED = ((TAIL + 1023) & ~1023) + 2 * S_TILE + 4 * 8 * HH * 4 + XU_TILE + WP_TILE;   // + M1 cache (M1C, declared below)
  static constexpr int NS_FIT = (SMEM_MAX - 2048 - FIXED) / STAGE;
  static constexpr int NS = NS_FIT < 2 * NSTEP ? NS_FIT : 2 * NSTEP;   // ring depth
  static constexpr int SMEM = 1024 + NS * STAGE + FIXED;
  static constexpr int CWF = HH / 4;                  // columns per epilogue thread
  static constexpr int M1C = 4 * REGT_F * HH * 4;     // bytes of the 4-slot cache of per-region M1 blocks
  static constexpr int TCOLS = 4 * HH;                // TMEM columns: A hi | A lo | acc0 | acc1
  static_assert(HH % 32 == 0 && TCOLS <= 512 && NS >= 3, "unsupported hidden width");
};

struct FArgs {
  int BN, BNp, N, T, nseg, mode, Bsz, nqt;
  const float *Xt, *St, *Ut;       // period-major F-wide features [T][rows][F]
  const int32_t *seg_ptr, *seg_reg;
  const float* M1t;                // [R][F][H] fp32 (region 0 is also in the image)
  const uint8_t* img;
  float *Zp, *Rp, *Hcp;            // saved planes, tile layout [T][nqt][H/4][128][4]
  float* out_hidden;               // [BN][H]
  int dbg;                         // 0: off; k > 0: record the phase timestamps of steps [k, k + 16) of CTA 0
  int save;                        // 0: forward only -- Z goes to a per-CTA scratch tile (Zp = [grid][128][H]), R and H~ nowhere
  // backward
  const float* G;                  // gradient wrt out_hidden, tile layout [nqt][H/4][128][4] (the head writes it that way)
  float *D, *hpl, *hRpl;           // transposed tiles [T*nqt][4 row quarters][4H | H | H][32 rows]
  double* dpp;                     // [grid][T] attention-gradient partials
  int hpre_mma;                    // forward: h_pre on the tensor cores where the item allows it (TEST HOOK REGT_F_HPRE_MMA=0: CUDA cores)
};

__device__ __forceinline__ uint32_t tf32_rn_bits(float a) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(a));
  return u;
}
__device__ __forceinline__ float sigm(float v) { return __fdividef(1.0f, 1.0f + __expf(-v)); }
__device__ __forceinline__ float tanh_(float v) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * v)); }

// 16 fp32 values of this thread's row -> tf32 hi | lo columns [col, col+16) of the TMEM A operand
template <int HH>
__device__ __forceinline__ void put_a16(uint32_t tlane, int col, const float (&v)[16]) {
  uint32_t hi[16], lo[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    hi[i] = tf32_rn_bits(v[i]);
    lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
  }
  tmem_st16(tlane + col, hi);
  tmem_st16(tlane + HH + col, lo);
}
template <int HH>
__device__ __forceinline__ void put_a8(uint32_t tlane, int col, const float (&v)[8]) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    hi[i] = tf32_rn_bits(v[i]);
    lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
  }
  tmem_st8(tlane + col, hi);
  tmem_st8(tlane + HH + col, lo);
}
__device__ __forceinline__ void st_f32x8(uint32_t taddr, const float (&v)[8]) {
  uint32_t u[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) u[i] = __float_as_uint(v[i]);
  tmem_st8(taddr, u);
}
template <int HH>
__device__ __forceinline__ void get_a16(uint32_t tlane, int col, float (&v)[16]) {
  float lo[16];
  tmem_ld16(tlane + col, v);
  tmem_ld16(tlane + HH + col, lo);
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] += lo[i];
}
// accumulator chunk + the A operand chunk (hi + lo) of the same 16 columns: three TMEM reads in flight, one wait
template <int HH>
__device__ __forceinline__ void get_acc_a16(uint32_t tacc, uint32_t tlane, int col, float (&v)[16], float (&h)[16]) {
  uint32_t rv[16], rh[16], rl[16];
  tmem_ld16_nw(tacc, rv);
  tmem_ld16_nw(tlane + col, rh);
  tmem_ld16_nw(tlane + HH + col, rl);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    v[i] = __uint_as_float(rv[i]);
    h[i] = __uint_as_float(rh[i]) + __uint_as_float(rl[i]);
  }
}
__device__ __forceinline__ void st_f32x16(uint32_t taddr, const float (&v)[16]) {
  uint32_t u[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) u[i] = __float_as_uint(v[i]);
  tmem_st16(taddr, u);
}

// byte offset of the 16-byte piece holding columns [c, c+4) of row r inside a saved-plane tile [H/4][128][4]
__device__ __forceinline__ size_t piece(int r, int c) { return ((size_t)(c >> 2) * TC_ROWS + r) * 16; }

struct Row {
  long long q;
  int b, s0, s1;
  bool valid;
  __device__ __forceinline__ void set(const FArgs& a, int qt, int r) {
    q = (long long)qt * TC_ROWS + r;
    valid = q < a.BN;
    b = valid ? (int)(q / a.N) : 0;
    s0 = s1 = 0;
    if (valid && a.mode != REGT_MODE_TGCN) {
      const int n = (int)(q - (long long)b * a.N);
      s0 = a.seg_ptr[n];
      s1 = a.seg_ptr[n + 1];
    }
  }
};

struct Feats {
  float x[8], u[8];
};
__device__ __forceinline__ void load8(const float* p, float (&v)[8], float m) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = m * a.x; v[1] = m * a.y; v[2] = m * a.z; v[3] = m * a.w; v[4] = m * b.x; v[5] = m * b.y; v[6] = m * b.z; v[7] = m * b.w;
}
__device__ __forceinline__ void load_feats(const FArgs& a, const Row& ri, int t, Feats& f) {
  const float m = ri.valid ? 1.f : 0.f;
  load8(a.Xt + ((size_t)t * a.BN + (ri.valid ? ri.q : 0)) * F, f.x, m);
  if (ri.s1 > ri.s0) load8(a.Ut + (((size_t)t * a.Bsz + ri.b) * a.nseg + ri.s0) * F, f.u, 1.f);
  else {
#pragma unroll
    for (int i = 0; i < 8; ++i) f.u[i] = 0.f;
  }
}
// h[16] for columns [c, c+16) of one row at period t: the regional combine on the F-wide features
// (models/RegionalTemporalGCN.py:136-143 collapsed: X_t M0 + sum_seg U_seg,t M1[region] + c0, leaky_relu)
// per-CTA cache of the M1 blocks of the regions a tile touches (shared memory, 4 direct-mapped slots keyed by region & 3):
// rows of a 128-row tile lie in one or two consecutive regions, so every lookup hits; anything else (a node in several
// regional lists, the random decomposition) falls back to the global copy
struct M1Cache {
  const float* data;      // [4][F][HH]
  const int* tag;         // [4] region held by the slot, -1 = empty
};
__device__ __forceinline__ void named_bar(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
// called by ALL epilogue threads at the first period of an item, with the row's first regional segment (or -1)
template <int HH>
__device__ __forceinline__ void m1_cache_fill(const FArgs& a, const Row& ri, float* data, int* tag, int etid) {
  constexpr int NEPI = NEPI_W * 32;
  if (a.mode != REGT_MODE_REGIONAL && a.nseg == 0) return;
  if (ri.s1 > ri.s0) {
    const int reg = a.seg_reg[ri.s0];
    tag[reg & 3] = reg;                 // racy on purpose: any row of the slot may win, the copy below uses the winner
  }
  named_bar(1, NEPI);
  constexpr int SLOT4 = F * HH / 4;     // float4 per slot
  for (int i = etid; i < 4 * SLOT4; i += NEPI) {
    const int slot = i / SLOT4, reg = tag[slot];
    if (reg >= 0)
      reinterpret_cast<float4*>(data)[i] = __ldg(reinterpret_cast<const float4*>(a.M1t) + (size_t)reg * SLOT4 + (i - slot * SLOT4));
  }
  named_bar(1, NEPI);
}
template <int HH, int NC>
__device__ __forceinline__ void hcols(const FArgs& a, const float* consts, const M1Cache& mc, const Row& ri, const Feats& f, int t, int c,
                                      float (&h)[NC]) {
  using C = FCfg<HH>;
#pragma unroll
  for (int i = 0; i < NC; ++i) h[i] = consts[C::C_C0 + c + i];
#pragma unroll
  for (int k = 0; k < F; ++k) {
#pragma unroll
    for (int i = 0; i < NC; i += 4) {
      const float4 w = *reinterpret_cast<const float4*>(consts + C::C_M0 + k * HH + c + i);
      h[i] = fmaf(f.x[k], w.x, h[i]); h[i + 1] = fmaf(f.x[k], w.y, h[i + 1]);
      h[i + 2] = fmaf(f.x[k], w.z, h[i + 2]); h[i + 3] = fmaf(f.x[k], w.w, h[i + 3]);
    }
  }
  for (int s = ri.s0; s < ri.s1; ++s) {
    const int reg = a.seg_reg[s];
    float uv[8];
    if (s == ri.s0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) uv[i] = f.u[i];
    } else {   // a node that appears in several regional lists (random decomposition)
      load8(a.Ut + (((size_t)t * a.Bsz + ri.b) * a.nseg + s) * F, uv, 1.f);
    }
    if (mc.tag[reg & 3] == reg) {
      const float* m = mc.data + (reg & 3) * F * HH + c;
#pragma unroll
      for (int k = 0; k < F; ++k) {
#pragma unroll
        for (int i = 0; i < NC; i += 4) {
          const float4 w = *reinterpret_cast<const float4*>(m + k * HH + i);
          h[i] = fmaf(uv[k], w.x, h[i]); h[i + 1] = fmaf(uv[k], w.y, h[i + 1]);
          h[i + 2] = fmaf(uv[k], w.z, h[i + 2]); h[i + 3] = fmaf(uv[k], w.w, h[i + 3]);
        }
      }
    } else {
      const float* m = a.M1t + (size_t)reg * F * HH + c;
#pragma unroll
      for (int k = 0; k < F; ++k) {
#pragma unroll
        for (int i = 0; i < NC; i += 4) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(m + k * HH + i));
          h[i] = fmaf(uv[k], w.x, h[i]); h[i + 1] = fmaf(uv[k], w.y, h[i + 1]);
          h[i + 2] = fmaf(uv[k], w.z, h[i + 2]); h[i + 3] = fmaf(uv[k], w.w, h[i + 3]);
        }
      }
    }
  }
  if (a.mode == REGT_MODE_REGIONAL) {
#pragma unroll
    for (int i = 0; i < NC; ++i) h[i] = h[i] > 0.f ? h[i] : 0.01f * h[i];   // F.leaky_relu
  }
}
template <int HH>
__device__ __forceinline__ void h16(const FArgs& a, const float* consts, const M1Cache& mc, const Row& ri, const Feats& f, int t, int c,
                                    float (&h)[16]) {
  hcols<HH, 16>(a, consts, mc, ri, f, t, c, h);
}

// one H x H block: acc (+)= A(TMEM, hi|lo) . W_g^T over the NCH ring stages of gate block g, three tf32 products
// (hi*hi + lo*hi + hi*lo).  Called by the whole MMA warp; lane 0 issues.
template <int HH>
__device__ __forceinline__ void mma_block(uint32_t tmem, uint32_t acc_col, uint32_t ring0, uint64_t* bar_full, uint64_t* bar_empty,
                                          long long& gs, int lane, bool accumulate, long long* wait_clk = nullptr) {
  using C = FCfg<HH>;
  const uint32_t idesc = make_idesc(FMT_TF32, 128, HH, 0, 0);
#pragma unroll 1
  for (int kc = 0; kc < C::NCH; ++kc, ++gs) {
    const int st = (int)(gs % C::NS);
    const long long w0 = wait_clk ? clock64() : 0;
    mbar_wait(&bar_full[st], (uint32_t)((gs / C::NS) & 1));
    if (wait_clk) *wait_clk += clock64() - w0;
    tc_fence_after();
    if (lane == 0) {
      const uint32_t bt = ring0 + st * C::STAGE;
#pragma unroll
      for (int p = 0; p < 3; ++p) {
        const uint32_t ap = tmem + (p == 1 ? HH : 0) + kc * 32, bp = bt + (p == 2 ? C::TILE : 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_ts_tf32(tmem + acc_col, ap + 8 * k, make_desc(bp + k * 32, 16, 1024, LAYOUT_SW128), idesc,
                       (accumulate || kc > 0 || p > 0 || k > 0) ? 1u : 0u);
      }
      umma_commit(&bar_empty[st]);   // the stage may be refilled once these MMAs have read it
    }
    __syncwarp();
  }
}
// the F-wide part of a gate: acc += S_t (smem chunk tile, hi|lo) . Ws_g^T   (K = 8: one MMA per product)
template <int HH>
__device__ __forceinline__ void mma_spart(uint32_t tmem, uint32_t acc_col, uint32_t stile, uint32_t sw_g, int lane) {
  using C = FCfg<HH>;
  if (lane == 0) {
    const uint32_t idesc = make_idesc(FMT_TF32, 128, HH, 0, 0);
#pragma unroll
    for (int p = 0; p < 3; ++p)
      umma<FMT_TF32>(tmem + acc_col, make_desc(stile + (p == 1 ? C::S_TILE : 0), TC_ROWS * 16, 128, LAYOUT_NONE),
                     make_desc(sw_g + (p == 2 ? C::SW_TILE : 0), HH * 16, 128, LAYOUT_NONE), idesc, 1u);
  }
  __syncwarp();
}

// F-wide features of one (tile, period) -> L2: 128 rows x 32 bytes of X_t (and S_t, and U_t where every node has exactly one
// regional segment in node order, as in the regional decomposition) are contiguous runs of the period-major arrays
__device__ __forceinline__ void prefetch_feats(const FArgs& a, int t, int qt) {
  const long long q0 = (long long)qt * TC_ROWS;
  const int rows = (int)min((long long)TC_ROWS, (long long)a.BN - q0);
  if (rows <= 0) return;
  const uint32_t bytes = (uint32_t)rows * F * 4;
  bulk_prefetch_l2(a.Xt + ((size_t)t * a.BN + q0) * F, bytes);
  bulk_prefetch_l2(a.St + ((size_t)t * a.BN + q0) * F, bytes);
  if (a.nseg == a.N) bulk_prefetch_l2(a.Ut + ((size_t)t * a.BN + q0) * F, bytes);   // segment of node n = n: same row order as X
}
// weight-stage producer: cycles the NSTEP stages of the image for every (tile, period) of this CTA
template <int HH>
__device__ __forceinline__ void produce(const uint8_t* img, uint8_t* ring, uint64_t* bar_full, uint64_t* bar_empty, long long total) {
  using C = FCfg<HH>;
  for (long long gs = 0; gs < total; ++gs) {
    const int st = (int)(gs % C::NS);
    if (gs >= C::NS) mbar_wait(&bar_empty[st], (uint32_t)((gs / C::NS - 1) & 1));
    mbar_arrive_expect_tx(&bar_full[st], C::STAGE);
    const uint8_t* src = img + (size_t)(gs % C::NSTEP) * C::STAGE;
#pragma unroll
    for (int o = 0; o < C::STAGE; o += 16384) bulk_g2s(ring + (size_t)st * C::STAGE + o, src + o, 16384, &bar_full[st]);
  }
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int HH>
__global__ void __launch_bounds__(NTHR, 1) k_cell_fwd_f(FArgs a) {
  using C = FCfg<HH>;
  constexpr int CWF = C::CWF;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = sm;
  uint8_t* tail = ring + C::NS * C::STAGE;                    // S-part weights | constants
  uint8_t* stile = tail + ((C::TAIL + 1023) & ~1023);         // S_t operand tile (hi | lo)
  float* m1data = reinterpret_cast<float*>(stile + 2 * C::S_TILE);
  uint8_t* xu = reinterpret_cast<uint8_t*>(m1data) + C::M1C;   // [3 k-steps][hi | lo] chunk tiles of [X | U(ra) | U(rb)]
  uint8_t* wp = xu + C::XU_TILE;                               // [3 k-steps][hi | lo] chunk tiles of [M0 ; M1[ra] ; M1[rb]]^T
  __shared__ uint64_t bar_full[C::NS], bar_empty[C::NS], bar_tail, bar_a, bar_z, bar_r, bar_a2, bar_c, bar_cfree, bar_x, bar_p;
  __shared__ uint32_t tmem_base_s;
  __shared__ int m1tag[4];
  __shared__ int pregs[2], pover, puse;    // the (at most two) regions of the item's rows, "does not fit" flag, path of the item
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_items = (a.nqt - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int S = n_items * a.T;

  if (tid == 0) {
    for (int s = 0; s < C::NS; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_tail, 1);
    mbar_init(&bar_a, NEPI_W * 32);
    mbar_init(&bar_z, 1);
    mbar_init(&bar_r, 1);
    mbar_init(&bar_a2, NEPI_W * 32);
    mbar_init(&bar_c, 1);
    mbar_init(&bar_cfree, NEPI_W * 32);
    mbar_init(&bar_x, NEPI_W * 32);
    mbar_init(&bar_p, 1);
    m1tag[0] = m1tag[1] = m1tag[2] = m1tag[3] = -1;
    puse = 0;
    fence_barrier_init();
    mbar_arrive_expect_tx(&bar_tail, C::TAIL);
    for (int o = 0; o < C::TAIL; o += 16384) bulk_g2s(tail + o, a.img + C::RING_IMG + o, min(16384, C::TAIL - o), &bar_tail);
  }
  if (warp == W_MMA) tmem_alloc(&tmem_base_s, C::TCOLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const float* consts = reinterpret_cast<const float*>(tail + C::SW_IMG);

  if (warp < NEPI_W) regs_grow(); else regs_shrink();
  if (warp < NEPI_W) {
    // ================= epilogue threads: thread = (row r = TMEM lane, CWF columns) =================
    mbar_wait(&bar_tail, 0);
    const int qd = warp & 3, ch = warp >> 2;
    const int r = qd * 32 + lane, c0 = ch * CWF;
    const uint32_t tl = tmem + ((uint32_t)(qd * 32) << 16);
    const uint32_t tZ = tl + 2 * HH, tR = tl + 3 * HH;
    float acc[CWF];
#pragma unroll
    for (int j = 0; j < CWF; ++j) acc[j] = 0.f;
    Row ri;
    const M1Cache mc{m1data, m1tag};
    // P(s) in two halves: Pcompute (h of step s on the CUDA cores, into registers; runs under the candidate MMAs of step
    // s - 1) and Pstore (registers -> TMEM A, S_t tile -> smem, bar_a; as soon as those MMAs have released A)
    // h of the next step waits in the (free) z-gate accumulator columns of TMEM, not in registers: next to acc[] it pushed the
    // epilogue warps over their 112 registers (ncu: 34 STL + 43 LDL per thread and step, through a 28 KB L1 into L2)
    float svn[8];
    // h_pre = X M0 + U M1[region] (+ c0, leaky_relu) of the NEXT step.  Regional mode, items whose rows lie in at most two
    // regions with one regional segment each (always, for the reference's contiguous regions of more than 64 nodes): ONE K = 24
    // MMA group  [X | U.1(r = ra) | U.1(r = rb)] . [M0 ; M1[ra] ; M1[rb]]  into the free z-accumulator columns -- the epilogue
    // threads only stage the 16 features of a row (ch 1: X, ch 2: U) instead of 512 FMAs per thread (4.2 of the 11.4 us of
    // epilogue work per step).  Other items: the CUDA-core sum, parked in the same columns.
    bool use_mma = false;
    int slot = -1;                            // this row's region slot (0 = ra, 1 = rb), -1: no regional segment
    constexpr int NEPI = NEPI_W * 32;
    auto Pcompute = [&](int s) {
      const int k = s / a.T, t = s - k * a.T;
      const int qt = (int)blockIdx.x + k * (int)gridDim.x;
      if (t == 0) {
        ri.set(a, qt, r);
        // every epilogue thread has finished the previous item's last Pcompute before any of them gets here (bar_a2 chain),
        // and the previous item's last h_pre MMAs have completed (bar_p was waited on in Pstore)
        const int nsg = ri.s1 - ri.s0;
        const int reg = nsg > 0 ? a.seg_reg[ri.s0] : -1;
        if (a.mode == REGT_MODE_REGIONAL && a.hpre_mma) {
          if (tid == 0) { pregs[0] = pregs[1] = -1; pover = 0; }
          named_bar(1, NEPI);
          if (ch == 0) {
            if (nsg > 1) pover = 1;
            else if (nsg == 1) {
              const int o0 = atomicCAS(&pregs[0], -1, reg);
              if (o0 != -1 && o0 != reg) {
                const int o1 = atomicCAS(&pregs[1], -1, reg);
                if (o1 != -1 && o1 != reg) pover = 1;
              }
            }
          }
          named_bar(1, NEPI);
          use_mma = pover == 0;
        } else {
          use_mma = false;
        }
        if (use_mma) {
          slot = nsg == 1 ? (pregs[0] == reg ? 0 : 1) : -1;
          // B operand of the item: element (k-step j, output n, kk) at chunk (kk >> 2) of row n, hi | lo
          for (int i = tid; i < 3 * F * HH; i += NEPI) {
            const int j = i / (F * HH), rem = i - j * (F * HH), kk = rem / HH, n = rem - kk * HH;
            float v;
            if (j == 0) v = consts[C::C_M0 + kk * HH + n];
            else {
              const int rg = pregs[j - 1];
              v = rg >= 0 ? __ldg(a.M1t + ((size_t)rg * F + kk) * HH + n) : 0.f;
            }
            const float hi = __uint_as_float(tf32_rn_bits(v));
            uint8_t* w0 = wp + j * 2 * C::SW_TILE + chunk_off(n, kk >> 2, HH) + (kk & 3) * 4;
            *reinterpret_cast<float*>(w0) = hi;
            *reinterpret_cast<float*>(w0 + C::SW_TILE) = v - hi;
          }
          if (tid == 0) puse = 1;
        } else {
          if (tid == 0) puse = 0;
          m1_cache_fill<HH>(a, ri, m1data, m1tag, tid);
        }
      }
      if (ch == 0) load8(a.St + ((size_t)t * a.BN + (ri.valid ? ri.q : 0)) * F, svn, ri.valid ? 1.f : 0.f);
      if (use_mma) {
        if (ch == 1 || ch == 2) {
          float v[8];
          const float m = ri.valid ? 1.f : 0.f;
          if (ch == 1) load8(a.Xt + ((size_t)t * a.BN + (ri.valid ? ri.q : 0)) * F, v, m);
          else if (slot >= 0) load8(a.Ut + (((size_t)t * a.Bsz + ri.b) * a.nseg + ri.s0) * F, v, m);
          else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0.f;
          }
          float hi[8], lo[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            hi[i] = __uint_as_float(tf32_rn_bits(v[i]));
            lo[i] = v[i] - hi[i];
          }
          const int j = ch == 1 ? 0 : (slot == 1 ? 2 : 1);      // k-step that receives this row's values
          uint8_t* t0 = xu + j * 2 * C::S_TILE;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            *reinterpret_cast<float4*>(t0 + chunk_off(r, c, TC_ROWS)) = make_float4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
            *reinterpret_cast<float4*>(t0 + C::S_TILE + chunk_off(r, c, TC_ROWS)) = make_float4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
          }
          if (ch == 2) {    // the other region slot of this row is zero
            uint8_t* z0 = xu + (j == 1 ? 2 : 1) * 2 * C::S_TILE;
            const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              *reinterpret_cast<float4*>(z0 + chunk_off(r, c, TC_ROWS)) = zero;
              *reinterpret_cast<float4*>(z0 + C::S_TILE + chunk_off(r, c, TC_ROWS)) = zero;
            }
          }
        }
        fence_proxy_async();
      } else {
        Feats f;
        load_feats(a, ri, t, f);
#pragma unroll
        for (int j = 0; j < CWF; j += 16) {
          float h[16];
          h16<HH>(a, consts, mc, ri, f, t, c0 + j, h);
          st_f32x16(tZ + c0 + j, h);     // acc_z is free here: E1z of this step has read it, the next z-gate MMAs wait for bar_a
        }
        tmem_st_wait();
      }
      tc_fence_before();
      mbar_arrive(&bar_x);               // operands staged (or h parked): the MMA warp issues the h_pre MMAs / passes on
    };
    int n_p = 0;                         // completed bar_p phases consumed
    auto Pstore = [&]() {
      if (ch == 0) {   // the F-wide gate operand S_t of this row: two 16-byte chunks, hi | lo
        float hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          hi[i] = __uint_as_float(tf32_rn_bits(svn[i]));
          lo[i] = svn[i] - hi[i];
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          *reinterpret_cast<float4*>(stile + chunk_off(r, c, TC_ROWS)) = make_float4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
          *reinterpret_cast<float4*>(stile + C::S_TILE + chunk_off(r, c, TC_ROWS)) = make_float4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
        }
        fence_proxy_async();
      }
      mbar_wait(&bar_p, (uint32_t)(n_p & 1));
      ++n_p;
      tc_fence_after();
#pragma unroll
      for (int j = 0; j < CWF; j += 16) {
        float h[16];
        tmem_ld16(tZ + c0 + j, h);
        if (use_mma) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float v = h[i] + consts[C::C_C0 + c0 + j + i];
            h[i] = v > 0.f ? v : 0.01f * v;          // F.leaky_relu of the regional combine
          }
        }
        put_a16<HH>(tl, c0 + j, h);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&bar_a);
    };
    if (S > 0) {
      Pcompute(0);
      Pstore();
    }
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      const int k = s / a.T, t = s - k * a.T;
      const int qt = (int)blockIdx.x + k * (int)gridDim.x;
      const long long q_cur = (long long)qt * TC_ROWS + r;
      const float p = consts[C::C_PROBS + t];
      const size_t toff = ((size_t)t * a.nqt + qt) * (size_t)(TC_ROWS * HH * 4);
      // forward only (inference): Z makes its round trip through a per-CTA tile that never leaves L2
      uint8_t* zt = reinterpret_cast<uint8_t*>(a.Zp) + (a.save ? toff : (size_t)blockIdx.x * (size_t)(TC_ROWS * HH * 4));
      uint8_t* rt = reinterpret_cast<uint8_t*>(a.Rp) + toff;
      uint8_t* ct = reinterpret_cast<uint8_t*>(a.Hcp) + toff;
      // ---- E1z: update gate (runs while the r-gate MMAs are in flight) ----
      F_TS(0, 0)
      mbar_wait(&bar_z, ph);
      tc_fence_after();
      F_TS(0, 1)
#pragma unroll
      for (int j = 0; j < CWF; j += 16) {
        float v[16], h[16];
        get_acc_a16<HH>(tZ + c0 + j, tl, c0 + j, v, h);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          v[i] = sigm(v[i] + consts[C::C_CZR + c0 + j + i]);
          acc[j + i] = fmaf(p * v[i], h[i], acc[j + i]);
        }
#pragma unroll
        for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(zt + piece(r, c0 + j + i)) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
      // ---- E1r: reset gate, h*R -> A operand of the candidate GEMM ----
      F_TS(0, 2)
      mbar_wait(&bar_r, ph);
      tc_fence_after();
      F_TS(0, 3)
#pragma unroll 1
      for (int j = 0; j < CWF; j += 16) {
        float v[16], h[16];
        get_acc_a16<HH>(tR + c0 + j, tl, c0 + j, v, h);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          v[i] = sigm(v[i] + consts[C::C_CZR + HH + c0 + j + i]);
          h[i] *= v[i];
        }
        put_a16<HH>(tl, c0 + j, h);
        if (a.save) {
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(rt + piece(r, c0 + j + i)) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&bar_a2);
      F_TS(0, 4)
      if (s + 1 < S) Pcompute(s + 1);      // under the candidate MMAs (h of the next step waits in registers)
      // ---- candidate GEMM done: A is free -> h of the next step goes in first (its z-gate MMAs start), then E2 under them ----
      F_TS(0, 5)
      mbar_wait(&bar_c, ph);
      tc_fence_after();
      F_TS(0, 6)
      if (s + 1 < S) Pstore();
      F_TS(0, 7)
#pragma unroll
      for (int j = 0; j < CWF; j += 16) {
        float v[16];
        float4 zq[4];
        // Z of this chunk: this thread's own stores of E1z, re-read with ordinary (coherent) loads -- all four issued before
        // any is used (one asm-volatile load per use serialised four L2 round trips per chunk: 2.4 us per step)
#pragma unroll
        for (int i = 0; i < 4; ++i) zq[i] = *reinterpret_cast<const float4*>(zt + piece(r, c0 + j + 4 * i));
        tmem_ld16(tR + c0 + j, v);
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float zz[4] = {zq[i >> 2].x, zq[i >> 2].y, zq[i >> 2].z, zq[i >> 2].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float hc = tanh_(v[i + e] + consts[C::C_CC + c0 + j + i + e]);
            v[i + e] = hc;
            acc[j + i + e] = fmaf(p * (1.0f - zz[e]), hc, acc[j + i + e]);
          }
          if (a.save) *reinterpret_cast<float4*>(ct + piece(r, c0 + j + i)) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(&bar_cfree);
      F_TS(0, 8)
      if (t + 1 == a.T) {   // item done: out_hidden = sum_t probs[t] H'_t
        if (q_cur < a.BN) {
          float* o = a.out_hidden + (size_t)q_cur * HH + c0;
#pragma unroll
          for (int j = 0; j < CWF; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
        }
#pragma unroll
        for (int j = 0; j < CWF; ++j) acc[j] = 0.f;
      }
    }
    tc_fence_before();
  } else if (warp == W_MMA) {
    mbar_wait(&bar_tail, 0);
    const uint32_t ring0 = smem_u32(ring), sw0 = smem_u32(tail), st0 = smem_u32(stile);
    const uint32_t xu0 = smem_u32(xu), wp0 = smem_u32(wp);
    const volatile int* puse_v = &puse;
    // h_pre of step s: [X | U(ra) | U(rb)] . [M0 ; M1[ra] ; M1[rb]] -> the z-accumulator columns (free between E1z of step s - 1
    // and the z-gate MMAs of step s), K = 3 x 8, three tf32 products each; items on the CUDA-core path only pass the barrier on
    auto pmma = [&](int s) {
      mbar_wait(&bar_x, (uint32_t)(s & 1));
      tc_fence_after();
      if (lane == 0) {
        if (*puse_v) {
          const uint32_t idesc = make_idesc(FMT_TF32, 128, HH, 0, 0);
#pragma unroll
          for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int p = 0; p < 3; ++p)
              umma<FMT_TF32>(tmem + 2 * HH, make_desc(xu0 + j * 2 * C::S_TILE + (p == 1 ? C::S_TILE : 0), TC_ROWS * 16, 128, LAYOUT_NONE),
                             make_desc(wp0 + j * 2 * C::SW_TILE + (p == 2 ? C::SW_TILE : 0), HH * 16, 128, LAYOUT_NONE), idesc,
                             (j > 0 || p > 0) ? 1u : 0u);
        }
        umma_commit(&bar_p);
      }
      __syncwarp();
    };
    long long gs = 0;
    if (S > 0) pmma(0);
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      long long wclk = 0;
      long long* wp_clk = a.dbg ? &wclk : nullptr;
      F_TSM(0)
      mbar_wait(&bar_a, ph);
      tc_fence_after();
      F_TSM(1)
      mma_block<HH>(tmem, 2 * HH, ring0, bar_full, bar_empty, gs, lane, false, wp_clk);
      mma_spart<HH>(tmem, 2 * HH, st0, sw0, lane);
      if (lane == 0) umma_commit(&bar_z);
      __syncwarp();
      F_TSM(2)
      if (s > 0) {   // acc_c of the previous step (same columns as acc_r) has been read
        mbar_wait(&bar_cfree, (uint32_t)((s - 1) & 1));
        tc_fence_after();
      }
      F_TSM(3)
      mma_block<HH>(tmem, 3 * HH, ring0, bar_full, bar_empty, gs, lane, false, wp_clk);
      mma_spart<HH>(tmem, 3 * HH, st0, sw0 + 2 * C::SW_TILE, lane);
      if (lane == 0) umma_commit(&bar_r);
      __syncwarp();
      F_TSM(4)
      mbar_wait(&bar_a2, ph);
      tc_fence_after();
      F_TSM(5)
      mma_block<HH>(tmem, 3 * HH, ring0, bar_full, bar_empty, gs, lane, false, wp_clk);
      mma_spart<HH>(tmem, 3 * HH, st0, sw0 + 4 * C::SW_TILE, lane);
      if (lane == 0) umma_commit(&bar_c);
      __syncwarp();
      F_TSM(6)
      if (s + 1 < S) pmma(s + 1);
      F_TSM(7)
      if (a.dbg && blockIdx.x == 0 && lane == 0 && s >= a.dbg && s < a.dbg + 16) g_f_dbg[2][(s - a.dbg) * 12 + 8] = wclk;
    }
    tc_fence_before();
  } else if (warp == W_PROD && lane == 0) {
    // weight stages, and two steps ahead of them the F-wide features of the coming (tile, period) into L2
    auto pf = [&](int s) {
      const int k = s / a.T, t = s - k * a.T;
      prefetch_feats(a, t, (int)blockIdx.x + k * (int)gridDim.x);
    };
    if (S > 0) pf(0);
    if (S > 1) pf(1);
    long long gs = 0;
    for (int s = 0; s < S; ++s) {
      if (s + 2 < S) pf(s + 2);
      for (int i = 0; i < C::NSTEP; ++i, ++gs) {
        const int st = (int)(gs % C::NS);
        if (gs >= C::NS) mbar_wait(&bar_empty[st], (uint32_t)((gs / C::NS - 1) & 1));
        mbar_arrive_expect_tx(&bar_full[st], C::STAGE);
        const uint8_t* src = a.img + (size_t)i * C::STAGE;
#pragma unroll
        for (int o = 0; o < C::STAGE; o += 16384) bulk_g2s(ring + (size_t)st * C::STAGE + o, src + o, 16384, &bar_full[st]);
      }
    }
  }
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, C::TCOLS);
}

// ------------------------------------------------------------------------------------------
// backward (data gradients; the weight gradients are row contractions over what this kernel writes)
// ------------------------------------------------------------------------------------------
// TMEM gives every epilogue thread one ROW (lane) of the tile, so a warp-wide access with "row per lane" into a ROW-major
// plane touches 32 different 128-byte lines.  v0 did exactly that (65 us per (tile, period): 32 LSU wavefronts and 32
// half-written sectors per store instruction), v1 transposed through per-warp shared-memory staging tiles (40 us, LSU pipe
// 61 % busy).  v2 (this one) stores what the weight-gradient contraction reads TRANSPOSED, per (tile, period):
//     DT [tp][4 row quarters][4H][32]   hT, hRT [tp][4][H][32]        (tp = t * nqt + qt; quarter = 32 rows = one warp's lanes)
// Lane = row makes every store of one column a contiguous 128-byte line -- and a [column][row] tile is exactly the K-major
// operand the row contraction wants (K = rows): gemm_tma.cu reads these tiles with plain TMA boxes and no transposing
// converters.  v2 issued those lines as 192 scalar st.global per thread and step: 8.5 of the 17.7 us of phase E0 were spent
// stalled on the store path (timed with the stores removed, tools/f_phases.py).  Staging the lines in per-warp
// shared-memory slots for the bulk-copy engine (cp.async.bulk shared -> global) measured slower (33.3 vs 29.8 us per step: a put
// waits for the engine to have read the slot used two puts ago); what did help is in profiles/r02_fused_phases.md.
template <int HH>
struct BCfg {   // shared-memory plan of the backward: ring | resident tail | M1 cache
  using C = FCfg<HH>;
  // Dz (then Dr) of the step: HH/4 values per epilogue thread that live from E0 to the Dr -> A conversion.  In registers, next
  // to E0's unrolled 16-column chunks, they pushed the epilogue warps far over their 112 registers (ncu: 62 STL + 94 LDL per
  // thread and step, 5 GB of spill traffic per launch through a 28 KB L1 into L2 -- a quarter of the kernel's L2 traffic, and
  // E0 is L2-bound: with a quarter of the CTAs it takes 11.6 us instead of 18.5).  The backward does not need a deep weight
  // ring (its MMAs wait for the epilogue, not for the weights): two of its stages pay for a [HH/4][512] plane in shared memory.
  static constexpr int DZS = NEPI_W * 32 * (HH / 4) * 4;
  static constexpr int FIXED = ((C::TAIL + 1023) & ~1023) + C::M1C + DZS;
  static constexpr int NS_FIT = (SMEM_MAX - 12288 - FIXED) / C::STAGE;
  static constexpr int NS = NS_FIT < 2 * C::NSTEP ? NS_FIT : 2 * C::NSTEP;
  static constexpr int SMEM = 1024 + NS * C::STAGE + FIXED;
  static_assert(NS >= 3, "backward ring too shallow");
};

template <int HH, int NS>
__device__ __forceinline__ void mma_block_n(uint32_t tmem, uint32_t acc_col, uint32_t ring0, uint64_t* bar_full, uint64_t* bar_empty,
                                            long long& gs, int lane, bool accumulate) {
  using C = FCfg<HH>;
  const uint32_t idesc = make_idesc(FMT_TF32, 128, HH, 0, 0);
#pragma unroll 1
  for (int kc = 0; kc < C::NCH; ++kc, ++gs) {
    const int st = (int)(gs % NS);
    mbar_wait(&bar_full[st], (uint32_t)((gs / NS) & 1));
    tc_fence_after();
    if (lane == 0) {
      const uint32_t bt = ring0 + st * C::STAGE;
#pragma unroll
      for (int p = 0; p < 3; ++p) {
        const uint32_t ap = tmem + (p == 1 ? HH : 0) + kc * 32, bp = bt + (p == 2 ? C::TILE : 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_ts_tf32(tmem + acc_col, ap + 8 * k, make_desc(bp + k * 32, 16, 1024, LAYOUT_SW128), idesc,
                       (accumulate || kc > 0 || p > 0 || k > 0) ? 1u : 0u);
      }
      umma_commit(&bar_empty[st]);
    }
    __syncwarp();
  }
}
// ONE K chunk (32 A columns) of an H x H block, gated on `ready` (the epilogue threads have staged exactly these A columns);
// `done`, if given, gets an arrive when the chunk's MMAs (and everything before them) have completed
template <int HH, int NS>
__device__ __forceinline__ void mma_chunk_n(uint32_t tmem, uint32_t acc_col, uint32_t ring0, uint64_t* bar_full, uint64_t* bar_empty,
                                            long long& gs, int lane, int kc, bool accumulate, uint64_t* ready, uint32_t parity,
                                            uint64_t* done) {
  using C = FCfg<HH>;
  const uint32_t idesc = make_idesc(FMT_TF32, 128, HH, 0, 0);
  mbar_wait(ready, parity);
  const int st = (int)(gs % NS);
  mbar_wait(&bar_full[st], (uint32_t)((gs / NS) & 1));
  tc_fence_after();
  if (lane == 0) {
    const uint32_t bt = ring0 + st * C::STAGE;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      const uint32_t ap = tmem + (p == 1 ? HH : 0) + kc * 32, bp = bt + (p == 2 ? C::TILE : 0);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        umma_ts_tf32(tmem + acc_col, ap + 8 * k, make_desc(bp + k * 32, 16, 1024, LAYOUT_SW128), idesc,
                     (accumulate || kc > 0 || p > 0 || k > 0) ? 1u : 0u);
    }
    umma_commit(&bar_empty[st]);
    if (done) umma_commit(done);
  }
  __syncwarp();
  ++gs;
}
template <int HH, int NS>
__device__ __forceinline__ void produce_n(const uint8_t* img, uint8_t* ring, uint64_t* bar_full, uint64_t* bar_empty, long long total) {
  using C = FCfg<HH>;
  for (long long gs = 0; gs < total; ++gs) {
    const int st = (int)(gs % NS);
    if (gs >= NS) mbar_wait(&bar_empty[st], (uint32_t)((gs / NS - 1) & 1));
    mbar_arrive_expect_tx(&bar_full[st], C::STAGE);
    const uint8_t* src = img + (size_t)(gs % C::NSTEP) * C::STAGE;
#pragma unroll
    for (int o = 0; o < C::STAGE; o += 16384) bulk_g2s(ring + (size_t)st * C::STAGE + o, src + o, 16384, &bar_full[st]);
  }
}

template <int HH>
__global__ void __launch_bounds__(NTHR, 1) k_cell_bwd_f(FArgs a) {
  using C = FCfg<HH>;
  using BC = BCfg<HH>;
  constexpr int NS = BC::NS;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = sm;
  uint8_t* tail = ring + NS * C::STAGE;
  float* m1data = reinterpret_cast<float*>(tail + ((C::TAIL + 1023) & ~1023));
  float* dzp = m1data + C::M1C / 4 + (threadIdx.x & (NEPI_W * 32 - 1));   // Dz plane [HH/4][512]: this thread's column
#define DZ(i) dzp[(i) * (NEPI_W * 32)]
  // per K chunk: A columns of the chunk staged (bar_a / bar_az / bar_ar, all epilogue threads), M2z MMAs of the chunk done (bar_2z)
  __shared__ uint64_t bar_full[NS], bar_empty[NS], bar_tail, bar_a[4], bar_1, bar_az[4], bar_2z[4], bar_ar[4], bar_2r;
  __shared__ uint32_t tmem_base_s;
  __shared__ int m1tag[4];
  __shared__ double red[NEPI_W][64];      // attention-gradient partials: fp64 sums (see below)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_items = (a.nqt - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int S = n_items * a.T;

  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_tail, 1);
    for (int c = 0; c < 4; ++c) {
      mbar_init(&bar_a[c], NEPI_W * 32);
      mbar_init(&bar_az[c], NEPI_W * 32);
      mbar_init(&bar_ar[c], NEPI_W * 32);
      mbar_init(&bar_2z[c], 1);
    }
    mbar_init(&bar_1, 1);
    mbar_init(&bar_2r, 1);
    m1tag[0] = m1tag[1] = m1tag[2] = m1tag[3] = -1;
    fence_barrier_init();
    mbar_arrive_expect_tx(&bar_tail, C::TAIL);
    for (int o = 0; o < C::TAIL; o += 16384) bulk_g2s(tail + o, a.img + C::RING_IMG + o, min(16384, C::TAIL - o), &bar_tail);
  }
  for (int i = tid; i < NEPI_W * 64; i += NTHR) (&red[0][0])[i] = 0.0;
  if (warp == W_MMA) tmem_alloc(&tmem_base_s, C::TCOLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const float* consts = reinterpret_cast<const float*>(tail + C::SW_IMG);

  if (warp < NEPI_W) regs_grow(); else regs_shrink();
  if (warp < NEPI_W) {
    mbar_wait(&bar_tail, 0);
    const int qd = warp & 3, ch = warp >> 2;
    const int r = qd * 32 + lane;
    // Column ownership is K-CHUNK-MAJOR: in trip j a thread works on columns [32 j + 8 ch, + 8), so that after trip j of all
    // threads the 32 columns of K chunk j are complete and the MMA warp can issue that chunk while the epilogue is in trip j + 1
    // (with [32 ch, + 32) per thread a block of MMAs could only start when the whole phase was over: 2.8 + 2.2 us of waiting per
    // step for the dHR and dhg blocks).
    constexpr int NTRIP = C::NCH;
    const int cb = 8 * ch;
    const uint32_t tl = tmem + ((uint32_t)(qd * 32) << 16);
    const uint32_t t1c = tl + 2 * HH, t2c = tl + 3 * HH;   // acc1 = dHR (then dHR * R), acc2 = p G Z + dhg
    Row ri;
    const M1Cache mc{m1data, m1tag};
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      const int k = s / a.T, t = s - k * a.T;
      const int qt = (int)blockIdx.x + k * (int)gridDim.x;
      if (t == 0) {
        ri.set(a, qt, r);
        m1_cache_fill<HH>(a, ri, m1data, m1tag, tid);   // all threads are past the previous item's E0 (bar_ar / bar_2r chain)
      }
      const float p = consts[C::C_PROBS + t];
      const size_t tp = (size_t)t * a.nqt + qt;
      const size_t toff = tp * (size_t)(TC_ROWS * HH * 4);
      const uint8_t* zt = reinterpret_cast<const uint8_t*>(a.Zp) + toff;
      const uint8_t* rt = reinterpret_cast<const uint8_t*>(a.Rp) + toff;
      const uint8_t* ct = reinterpret_cast<const uint8_t*>(a.Hcp) + toff;
      const uint8_t* gt = reinterpret_cast<const uint8_t*>(a.G) + (size_t)qt * (size_t)(TC_ROWS * HH * 4);   // G tile of this item
      // transposed outputs of this (tile, period), this warp's row quarter: column c at c * 32 (+ lane)
      float* DT = a.D + (tp * 4 + qd) * (size_t)(4 * HH * 32);
      float* hT = a.hpl + (tp * 4 + qd) * (size_t)(HH * 32);
      float* hRT = a.hRpl + (tp * 4 + qd) * (size_t)(HH * 32);
      // ---- E0: recompute h; gate gradients from the saved planes ----
      F_TS(1, 0)
      Feats f;
      load_feats(a, ri, t, f);
      double dp = 0.0;
      unsigned int neg = 0u;                     // h <= 0 per column (leaky_relu slope of the regional combine)
      // Eight columns per trip of a ROLLED loop: the plane loads of the trip go first, h of the eight columns is recomputed under
      // them, every result leaves before the next trip (Dz -> shared memory, Dc -> A, p G Z -> acc2, h / hR / Dc / Dz -> their
      // transposed tiles).  Unrolled over 16-column chunks the compiler kept up to 16 float4 loads and five 16-column arrays
      // alive at once and spilled (see BCfg).
#pragma unroll 1
      for (int j = 0; j < NTRIP; ++j) {
        const int c = 32 * j + cb;
        float4 zq[2], rq[2], cq[2], gq[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          zq[i] = __ldcs(reinterpret_cast<const float4*>(zt + piece(r, c + 4 * i)));   // Z and H~ are read once: streaming loads
          cq[i] = __ldcs(reinterpret_cast<const float4*>(ct + piece(r, c + 4 * i)));
          rq[i] = __ldg(reinterpret_cast<const float4*>(rt + piece(r, c + 4 * i)));
          gq[i] = __ldg(reinterpret_cast<const float4*>(gt + piece(r, c + 4 * i)));
        }
        float h[8];
        hcols<HH, 8>(a, consts, mc, ri, f, t, c, h);
        if (j == 0) { F_TS(1, 9) }
        float dc[8], gz[8];
        float dpc = 0.f;
        unsigned int ng = 0u;
        float* o_h = hT + (size_t)c * 32 + lane;
        float* o_hr = hRT + (size_t)c * 32 + lane;
        float* o_dz = DT + (size_t)c * 32 + lane;
        float* o_dc = DT + (size_t)(2 * HH + c) * 32 + lane;
#pragma unroll
        for (int i = 0; i < 8; i += 4) {
          const float4 z4 = zq[i >> 2], r4 = rq[i >> 2], c4 = cq[i >> 2], g4 = gq[i >> 2];
          const float z[4] = {z4.x, z4.y, z4.z, z4.w}, rg[4] = {r4.x, r4.y, r4.z, r4.w}, hc[4] = {c4.x, c4.y, c4.z, c4.w};
          const float g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float hh = h[i + e];
            const float gv = ri.valid ? g[e] : 0.f;                           // padded rows of the last tile: zero gradient
            const float gg = p * gv;                                          // dH' = probs[t] * d out_hidden
            dpc = fmaf(gv, z[e] * hh + (1.0f - z[e]) * hc[e], dpc);
            const float dzv = gg * (hh - hc[e]) * z[e] * (1.0f - z[e]);
            dc[i + e] = gg * (1.0f - z[e]) * (1.0f - hc[e] * hc[e]);
            gz[i + e] = gg * z[e];
            DZ(8 * j + i + e) = dzv;
            if (!(hh > 0.f)) ng |= 1u << (i + e);
            o_h[(i + e) * 32] = hh;                                           // re-read in E1: not streamed
            __stcs(o_hr + (i + e) * 32, hh * rg[e]);                          // the other planes: streaming (evict-first) stores
            __stcs(o_dz + (i + e) * 32, dzv);
            __stcs(o_dc + (i + e) * 32, dc[i + e]);
          }
        }
        neg |= ng << (8 * j);
        dp += (double)dpc;
        if (j == 0) { F_TS(1, 10) }
        put_a8<HH>(tl, c, dc);
        st_f32x8(t2c + c, gz);                    // acc2 starts from p G Z: the dhg MMAs accumulate on top of it
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&bar_a[j]);                   // K chunk j of Dc is staged: its dHR MMAs run under the next trip
        if (j == 0) { F_TS(1, 11) }
      }
      F_TS(1, 1)
      // attention gradient d probs[t] += sum G * H'_t.  The softmax Jacobian takes differences of these nearly equal sums
      // (models/RegionalTemporalGCN.py:134), so everything above 16 terms is summed in fp64: fixed-order warp sum, one
      // shared-memory slot per (warp, period)
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) dp += __shfl_xor_sync(0xffffffffu, dp, d);
      if (lane == 0) red[warp][t] += dp;
      // ---- M1 done (dHR in acc1): Dz -> A chunk by chunk, M2z follows the chunks ----
      mbar_wait(&bar_1, ph);
      tc_fence_after();
      F_TS(1, 2)
#pragma unroll
      for (int j = 0; j < NTRIP; ++j) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = DZ(8 * j + i);
        put_a8<HH>(tl, 32 * j + cb, v);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&bar_az[j]);
      }
      F_TS(1, 3)
      // ---- E1 (under M2z): Dr = dHR h R (1-R), t1 = dHR R -> acc1 in place; as soon as the M2z MMAs of K chunk j have read A,
      //      Dr of that chunk goes in and its M2r MMAs follow ----
      __syncwarp();       // the h lines of E0 (this warp's own stores) are re-read below with ordinary loads
#pragma unroll 1
      for (int j = 0; j < NTRIP; ++j) {
        const int c = 32 * j + cb;
        float v[8], hh[8], dr[8];
        float4 rq[2];
#pragma unroll
        for (int i = 0; i < 8; ++i) hh[i] = hT[(size_t)(c + i) * 32 + lane];
#pragma unroll
        for (int i = 0; i < 2; ++i) rq[i] = __ldg(reinterpret_cast<const float4*>(rt + piece(r, c + 4 * i)));
        tmem_ld8(t1c + c, v);
        float* o_dr = DT + (size_t)(HH + c) * 32 + lane;
#pragma unroll
        for (int i = 0; i < 8; i += 4) {
          const float rg[4] = {rq[i >> 2].x, rq[i >> 2].y, rq[i >> 2].z, rq[i >> 2].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            dr[i + e] = v[i + e] * hh[i + e] * rg[e] * (1.0f - rg[e]);
            v[i + e] *= rg[e];
            __stcs(o_dr + (i + e) * 32, dr[i + e]);
          }
        }
        st_f32x8(t1c + c, v);
        mbar_wait(&bar_2z[j], ph);                // A columns of chunk j are free (Dz of the chunk has been consumed)
        tc_fence_after();
        put_a8<HH>(tl, c, dr);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&bar_ar[j]);
      }
      F_TS(1, 4)
      F_TS(1, 5)
      F_TS(1, 6)
      // ---- E2: d h_pre = act'(h) (p G Z + dhg + dHR R) ----
      mbar_wait(&bar_2r, ph);
      tc_fence_after();
      F_TS(1, 7)
#pragma unroll 1
      for (int j = 0; j < NTRIP; ++j) {
        const int c = 32 * j + cb;
        float v[8], u[8];
        tmem_ld8(t2c + c, v);
        tmem_ld8(t1c + c, u);
        float* o_dh = DT + (size_t)(3 * HH + c) * 32 + lane;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float d = v[i] + u[i];
          if (a.mode == REGT_MODE_REGIONAL && ((neg >> (8 * j + i)) & 1u)) d *= 0.01f;
          __stcs(o_dh + i * 32, d);
        }
      }
      tc_fence_before();
      F_TS(1, 8)
    }
  } else if (warp == W_MMA) {
    const uint32_t ring0 = smem_u32(ring);
    long long gs = 0;
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      // dHR = Dc . B_h, chunk by chunk behind E0 (bar_a[0] also says: E2 of the previous step has read acc1 / acc2)
      for (int kc = 0; kc < C::NCH; ++kc) mma_chunk_n<HH, NS>(tmem, 2 * HH, ring0, bar_full, bar_empty, gs, lane, kc, false, &bar_a[kc], ph, nullptr);
      if (lane == 0) umma_commit(&bar_1);
      __syncwarp();
      // acc2 = p G Z + Dz . B_z; every chunk reports its completion: E1 refills A with Dr of that chunk
      for (int kc = 0; kc < C::NCH; ++kc) mma_chunk_n<HH, NS>(tmem, 3 * HH, ring0, bar_full, bar_empty, gs, lane, kc, true, &bar_az[kc], ph, &bar_2z[kc]);
      // acc2 += Dr . B_r
      for (int kc = 0; kc < C::NCH; ++kc) mma_chunk_n<HH, NS>(tmem, 3 * HH, ring0, bar_full, bar_empty, gs, lane, kc, true, &bar_ar[kc], ph, nullptr);
      if (lane == 0) umma_commit(&bar_2r);
      __syncwarp();
    }
    tc_fence_before();
  } else if (warp == W_PROD && lane == 0) {
    // weight stages, and one step ahead of them the saved-plane tiles of the NEXT step into L2: the epilogue threads read
    // Z, R, H~ (and G once per item) with ordinary loads, which would otherwise wait out a DRAM round trip per 16-column chunk
    constexpr uint32_t TB = TC_ROWS * HH * 4;
    auto prefetch_step = [&](int s) {
      const int k = s / a.T, t = s - k * a.T;
      const int qt = (int)blockIdx.x + k * (int)gridDim.x;
      const size_t toff = ((size_t)t * a.nqt + qt) * (size_t)TB;
      bulk_prefetch_l2(reinterpret_cast<const uint8_t*>(a.Zp) + toff, TB);
      bulk_prefetch_l2(reinterpret_cast<const uint8_t*>(a.Rp) + toff, TB);
      bulk_prefetch_l2(reinterpret_cast<const uint8_t*>(a.Hcp) + toff, TB);
      if (t == 0) bulk_prefetch_l2(reinterpret_cast<const uint8_t*>(a.G) + (size_t)qt * TB, TB);
      prefetch_feats(a, t, qt);
    };
    // L2 prefetch of the next step's planes when the dHR MMAs of step s complete (bar_1), i.e. 6-8 us before E0 of step s + 1
    // reads them.  A whole step ahead (as the weight stages are issued) measured harmful: at 148 x 576 KB of plane traffic per
    // step the lines are evicted again before their step comes and DRAM reads double (ncu: 7.6 GB against 3.3 GB per launch).
    long long gs = 0;
    for (int s = 0; s < S; ++s) {
      bool pf_pending = s + 1 < S;
      for (int i = 0; i < C::NSTEP; ++i, ++gs) {
        const int st = (int)(gs % NS);
        if (gs >= NS) {
          const uint32_t par = (uint32_t)((gs / NS - 1) & 1);
          while (!mbar_try_wait(&bar_empty[st], par)) {
            if (pf_pending && mbar_try_wait(&bar_1, (uint32_t)(s & 1))) {
              prefetch_step(s + 1);
              pf_pending = false;
            }
          }
        }
        mbar_arrive_expect_tx(&bar_full[st], C::STAGE);
        const uint8_t* src = a.img + (size_t)i * C::STAGE;
#pragma unroll
        for (int o = 0; o < C::STAGE; o += 16384) bulk_g2s(ring + (size_t)st * C::STAGE + o, src + o, 16384, &bar_full[st]);
      }
      if (pf_pending) {      // all stages of the step were issued before its dHR MMAs finished
        mbar_wait(&bar_1, (uint32_t)(s & 1));
        prefetch_step(s + 1);
      }
    }
  }
  __syncthreads();
  if (tid < a.T) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < NEPI_W; ++w) s += red[w][tid];
    a.dpp[(size_t)blockIdx.x * a.T + tid] = s;
  }
  if (warp == W_MMA) tmem_dealloc(tmem, C::TCOLS);
}

// ------------------------------------------------------------------------------------------
// per-step weight images (forward: [S|h] gate weights; backward: B_g transposed for the data gradients)
// ------------------------------------------------------------------------------------------
template <int HH>
__device__ __forceinline__ void put_stage(uint8_t* img, int g, int n, int k, float v) {
  using C = FCfg<HH>;
  uint8_t* st = img + (size_t)(g * C::NCH + (k >> 5)) * C::STAGE;
  const uint32_t off = sw128_off(n, (k & 31) * 4, HH);
  const float hi = __uint_as_float(tf32_rn_bits(v));
  *reinterpret_cast<float*>(st + off) = hi;
  *reinterpret_cast<float*>(st + C::TILE + off) = v - hi;
}
// Wzr [F+H][2H], Wc [F+H][H] (rows 0..F-1: S part, rows F..: h part); lin_w[g] [H][2H]
template <int HH>
__global__ void k_pack_f(const float* __restrict__ Wzr, const float* __restrict__ Wc, const float* __restrict__ czr,
                         const float* __restrict__ cc, const float* __restrict__ c0, const float* __restrict__ M0t,
                         const float* __restrict__ M1t, const float* __restrict__ probs, int T, const float* __restrict__ lw0,
                         const float* __restrict__ lw1, const float* __restrict__ lw2, uint8_t* __restrict__ img_f,
                         uint8_t* __restrict__ img_b) {
  using C = FCfg<HH>;
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < 3 * HH * HH) {      // forward H-wide part: gate g, output n, input k
    const int g = j / (HH * HH), rem = j % (HH * HH), n = rem / HH, k = rem % HH;
    const float v = g < 2 ? Wzr[(size_t)(F + k) * 2 * HH + g * HH + n] : Wc[(size_t)(F + k) * HH + n];
    put_stage<HH>(img_f, g, n, k, v);
    // backward: dHR = Dc . B_h, dhg = Dz . B_z + Dr . B_r  ->  stage order  B_h, B_z, B_r ; tile rows = input index k_in,
    // K = gate output index:  Bt_g[k_in][n_out] = linear_g.weight[n_out][H + k_in]
    const int gb = (g == 0) ? 1 : (g == 1 ? 2 : 0);     // this thread's g indexes lw: z -> slot 1, r -> slot 2, h -> slot 0
    const float* lw = g == 0 ? lw0 : (g == 1 ? lw1 : lw2);
    put_stage<HH>(img_b, gb, /*row k_in=*/n, /*K index n_out=*/k, lw[(size_t)k * 2 * HH + HH + n]);
    return;
  }
  j -= 3 * HH * HH;
  if (j < 3 * HH * 8) {       // forward F-wide part: chunk tile [2][HH][16 B] per gate, hi | lo
    const int g = j / (HH * 8), rem = j % (HH * 8), n = rem / 8, f = rem % 8;
    const float v = g < 2 ? Wzr[(size_t)f * 2 * HH + g * HH + n] : Wc[(size_t)f * HH + n];
    uint8_t* t0 = img_f + C::RING_IMG + (size_t)g * 2 * C::SW_TILE;
    const uint32_t off = chunk_off(n, f >> 2, HH) + (f & 3) * 4;
    const float hi = __uint_as_float(tf32_rn_bits(v));
    *reinterpret_cast<float*>(t0 + off) = hi;
    *reinterpret_cast<float*>(t0 + C::SW_TILE + off) = v - hi;
    return;
  }
  j -= 3 * HH * 8;
  if (j < C::C_FLOATS) {
    float v = 0.f;
    if (j < C::C_CC) v = czr[j];
    else if (j < C::C_C0) v = cc[j - C::C_CC];
    else if (j < C::C_M0) v = c0 ? c0[j - C::C_C0] : 0.f;
    else if (j < C::C_M1) v = M0t ? M0t[j - C::C_M0] : 0.f;
    else if (j < C::C_PROBS) v = M1t ? M1t[j - C::C_M1] : 0.f;
    else v = (j - C::C_PROBS) < T ? probs[j - C::C_PROBS] : 0.f;
    reinterpret_cast<float*>(img_f + C::RING_IMG + C::SW_IMG)[j] = v;
    reinterpret_cast<float*>(img_b + C::RING_IMG + C::SW_IMG)[j] = v;
  }
}

// F^T tiles of the weight-gradient contraction, [tp][4 row quarters][32][32 rows]: rows 0..7 = S_t, 8..15 = X_t, 16 = 1, 17..31 = 0 of the 128 rows
// of tile tp = t * nqt + qt (padded rows q >= BN: all zero).  One thread per (tile, row): its 32-byte S and X rows are
// contiguous across the warp, every store of one feature is a 128-byte line.
__global__ void __launch_bounds__(128) k_featT_f(const float* __restrict__ Xt, const float* __restrict__ St, int BN, int nqt,
                                                 float* __restrict__ FT) {
  const int tp = blockIdx.x, r = threadIdx.x;
  const int t = tp / nqt, qt = tp - t * nqt;
  const long long q = (long long)qt * TC_ROWS + r;
  const bool ok = q < BN;
  float s[8], x[8];
  load8(St + ((size_t)t * BN + (ok ? q : 0)) * F, s, ok ? 1.f : 0.f);
  load8(Xt + ((size_t)t * BN + (ok ? q : 0)) * F, x, ok ? 1.f : 0.f);
  float* o = FT + ((size_t)tp * 4 + (r >> 5)) * (32 * 32) + (r & 31);      // [tp][row quarter][32 features][32 rows]
#pragma unroll
  for (int f = 0; f < 8; ++f) {
    o[(size_t)f * 32] = s[f];
    o[(size_t)(8 + f) * 32] = x[f];
  }
  o[(size_t)16 * 32] = ok ? 1.f : 0.f;
#pragma unroll
  for (int f = 17; f < 32; ++f) o[(size_t)f * 32] = 0.f;
}
// the head's weight-gradient contraction (head.cu) takes its bias column sums from a ones column: Feat [BNp][32], column 16
__global__ void __launch_bounds__(256) k_ones_f(int BN, int BNp, float* __restrict__ Feat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= BNp * 8) return;
  const int row = i >> 3, c4 = i & 7;
  reinterpret_cast<float4*>(Feat)[i] = make_float4((c4 == 4 && row < BN) ? 1.f : 0.f, 0.f, 0.f, 0.f);
}

template <int HH>
FArgs make_fargs(const regt_args* a, const Layout& L) {
  FArgs k{};
  k.BN = a->B * a->N; k.N = a->N; k.T = a->T; k.nseg = a->plan.nseg; k.mode = a->mode; k.Bsz = a->B;
  k.nqt = (k.BN + TC_ROWS - 1) / TC_ROWS;
  k.BNp = k.nqt * TC_ROWS;
  k.Xt = L.Xt; k.St = L.S; k.Ut = L.U;
  k.seg_ptr = a->plan.seg_ptr; k.seg_reg = a->plan.seg_reg;
  k.M1t = L.M1t;
  k.Zp = L.Zp; k.Rp = L.Rp; k.Hcp = L.Hcp;
  k.out_hidden = a->out_hidden;
  k.save = a->inference ? 0 : 1;
  {
    const char* e = getenv("REGT_F_DEBUG");
    k.dbg = e ? atoi(e) : 0;
    const char* hm = getenv("REGT_F_HPRE_MMA");     // read per launch: the test toggles it inside one process
    k.hpre_mma = !(hm && hm[0] == '0');
  }
  k.G = L.G; k.D = L.D; k.hpl = L.h; k.hRpl = L.hR; k.dpp = reinterpret_cast<double*>(L.tc_dpp);
  return k;
}

template <int HH>
int run_fwd(const regt_args* a, const Layout& L, cudaStream_t st) {
  using C = FCfg<HH>;
  static_assert(C::IMG <= F_IMG_BYTES, "weight image too large");
  const int n_pack = 3 * HH * HH + 3 * HH * 8 + C::C_FLOATS;
  k_pack_f<HH><<<cdiv(n_pack, 256), 256, 0, st>>>(L.Wzr, L.Wc, L.czr, L.cc, L.c0, L.M0t, L.M1t, L.probs, a->T, a->p.lin_w[0],
                                                  a->p.lin_w[1], a->p.lin_w[2], L.tc_img_f, L.tc_img_b);
  REGT_LAUNCHED("k_pack_f", st);
  return 0;
}
template <int HH>
int run_fwd_kernel(const regt_args* a, const Layout& L, cudaStream_t st) {
  using C = FCfg<HH>;
  FArgs k = make_fargs<HH>(a, L);
  k.img = L.tc_img_f;
  REGT_CUDA(cudaFuncSetAttribute(k_cell_fwd_f<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
  const int grid = min(sm_count(), k.nqt);
  REGT_CHECK(grid <= TC_MAX_CTAS, "fused forward: grid %d exceeds the per-CTA scratch tiles", grid);
  k_cell_fwd_f<HH><<<grid, NTHR, C::SMEM, st>>>(k);
  REGT_LAUNCHED("k_cell_fwd_f", st);
  return 0;
}
template <int HH>
int run_bwd_kernel(const regt_args* a, const Layout& L, cudaStream_t st, int* grid_out) {
  using C = FCfg<HH>;
  FArgs k = make_fargs<HH>(a, L);
  k.img = L.tc_img_b;
  const int grid = min(sm_count(), k.nqt);
  REGT_CHECK(grid <= TC_MAX_CTAS, "fused backward: grid %d exceeds the partial buffers", grid);
  REGT_CUDA(cudaFuncSetAttribute(k_cell_bwd_f<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, BCfg<HH>::SMEM));
  k_cell_bwd_f<HH><<<grid, NTHR, BCfg<HH>::SMEM, st>>>(k);
  REGT_LAUNCHED("k_cell_bwd_f", st);
  *grid_out = grid;
  return 0;
}
int launch_feat_f(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int BN = a->B * a->N, nqt = (BN + TC_ROWS - 1) / TC_ROWS, BNp = nqt * TC_ROWS;
  k_featT_f<<<a->T * nqt, 128, 0, st>>>(L.Xt, L.S, BN, nqt, L.FeatT);
  REGT_LAUNCHED("k_featT_f", st);
  k_ones_f<<<cdiv((long long)BNp * 8, 256), 256, 0, st>>>(BN, BNp, L.Feat);
  REGT_LAUNCHED("k_ones_f", st);
  return 0;
}
}  // namespace

bool cell_f_fits(const regt_args* a) { return (a->H == 128 || a->H == 64) && a->mode != REGT_MODE_TGCN && a->T <= 64; }

int cell_forward_f(const regt_args* a, const Layout& L, cudaStream_t st) {
  // features (graph + x) and collapsed weights (parameters) are independent: two streams
  cudaStream_t side = fork_side(st);
  cudaStream_t fs = side ? side : st;
  if (launch_feat_tc(a->plan, a->x, feat_in(a), a->B, a->x_rows > 0 ? a->x_rows : a->N, a->T, L.Xt, L.S, L.U, fs)) return -1;
  if (!a->inference && launch_feat_f(a, L, fs)) return -1;   // feature plane of the weight-gradient contractions (cell and head backward)
  if (launch_prep(a, L, st)) return -1;
  if (a->H == 128 ? run_fwd<128>(a, L, st) : run_fwd<64>(a, L, st)) return -1;
  if (side && join_side(st)) return -1;
  return a->H == 128 ? run_fwd_kernel<128>(a, L, st) : run_fwd_kernel<64>(a, L, st);
}

int cell_backward_f(const regt_args* a, const Layout& L, cudaStream_t st) {
  const int H = a->H, T = a->T;
  const long long BN = (long long)a->B * a->N, nqt = (BN + 127) / 128, ntile = nqt * T;
  int grid = 0;
  if (H == 128 ? run_bwd_kernel<128>(a, L, st, &grid) : run_bwd_kernel<64>(a, L, st, &grid)) return -1;
  if (launch_f_sum_dpp(reinterpret_cast<const double*>(L.tc_dpp), grid, T, L.dprobs, st)) return -1;
  // weight gradients: ONE row contraction over the transposed gate-gradient tiles D^T [tile][4H][128] (z | r against h,
  // h~ against h*R, h_pre against the feature tile only; every block also against [S | X | 1]), rows = K
  float* part = L.part;
  const int mtiles = 4 * H / 128;
  const int splits = (int)max(1ll, min((long long)min(WGRAD_SPLITS, cdiv(148, mtiles)), ntile / 4));
  float* pB = part;                                          // [splits][2H][H]  dB_z | dB_r
  float* pBh = pB + (size_t)splits * 2 * H * H;              // [splits][H][H]   dB_h
  float* pF = pBh + (size_t)splits * H * H;                  // [splits][4H][32] D^T Feat
  const long long fsplit = 4ll * H * 32;
  {
    // segments start at multiples of 128 columns.  H = 128: z|r (2 tiles), h~, h_pre.  H = 64: tile 0 = z|r, tile 1 = h~ | h_pre
    // (its rows 64.. are contracted against h*R too and dropped: only the feature columns of h_pre are kept)
    int k0[3], k1[3], sb[3];
    float* cs[3];
    int ns;
    if (H == 128) {
      ns = 3;
      k0[0] = 0; k1[0] = 256; sb[0] = 0; cs[0] = pB;
      k0[1] = 256; k1[1] = 384; sb[1] = 1; cs[1] = pBh;
      k0[2] = 384; k1[2] = 512; sb[2] = -1; cs[2] = nullptr;
    } else {
      ns = 2;
      k0[0] = 0; k1[0] = 128; sb[0] = 0; cs[0] = pB;
      k0[1] = 128; k1[1] = 192; sb[1] = 1; cs[1] = pBh;
    }
    const float* bs[2] = {L.h, L.hR};
    if (launch_gemm_kt(L.D, ntile, 4 * H, ns, k0, k1, sb, cs, bs, H, splits, L.FeatT, pF, fsplit, st)) return -1;
  }
  if (launch_reduce_splits(pB, L.dB, 2ll * H * H, splits, 0, st)) return -1;
  if (launch_reduce_splits(pBh, L.dB + (size_t)2 * H * H, (long long)H * H, splits, 0, st)) return -1;
  if (launch_fw_scatter(pF, splits, H, L, st)) return -1;
  if (a->plan.nseg > 0) {   // dM1[r]: per-region sums over the (node, region) segments
    if (launch_wgrad_m1_kt(a, L, st)) return -1;
  }
  return launch_chain(a, L, st);
}

}  // namespace regt

// TEST HOOK: phase timestamps (clock64) of the fused kernels, recorded when REGT_F_DEBUG=<first step> is set:
// out[which][step][mark], which 0 = forward, 1 = backward, 16 steps x 12 marks each
extern "C" int regt_debug_f_timestamps(long long* out) {
  REGT_CUDA(cudaMemcpyFromSymbol(out, regt::g_f_dbg, sizeof(long long) * 3 * 16 * 12));
  return 0;
}
