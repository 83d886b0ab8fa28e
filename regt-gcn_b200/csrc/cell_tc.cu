// tcgen05 (sm_100a tensor core) kernels of the regional temporal GCN cell.
//
// One persistent CTA per SM.  A work item is 128 rows (b,n) x a chunk of `tp` periods; thread r of
// the 256 epilogue threads owns row r (= TMEM lane r) and one half of the H columns, and walks the
// periods of its item, so the period-attention sum  sum_t probs[t] * H'_t  stays in registers.
// Per period:
//   P   CUDA cores : h = act(X_t M0 + U_t M1[r] + c0)  -> bf16 SW128 operand tile in smem
//   M1  tcgen05.mma: [S_t | h] x Wzr  -> TMEM cols [0,2H)          (weights resident in smem)
//   E1  CUDA cores : Z,R = sigmoid(. + czr) (tcgen05.ld), save Z,R; h*R -> operand tile
//   M2  tcgen05.mma: [S_t | h*R] x Wc -> TMEM cols [2H,3H)
//   E2  CUDA cores : H~ = tanh(. + cc), save H~;  acc += probs[t] * (Z h + (1-Z) H~)
// Precision: REGT_PREC_BF16 = bf16 operands, fp32 accumulate.
// Reference arithmetic replaced: models/utils.py:168-188 + models/RegionalTemporalGCN.py:134-148.
#include "cell_tc.cuh"
#include "gemm_simt.cuh"

// Pipeline variants measured on B200 at config 2 and dropped (profiles/r01_ab_variants.txt): a software-pipelined forward
// epilogue (47.0 against 38.5 us), h of step s+1 produced under M2 of step s in the backward (no gain), 16 columns per
// epilogue thread, one mbarrier arrival per warp.

namespace regt {
using namespace tc;
constexpr int F = REGT_F;
constexpr int CW = 32;                     // columns owned by one epilogue thread
constexpr int NEPI_WARPS = 4 * (64 / CW);  // 4 lane quarters x column groups (hidden = 64)
constexpr int NEPI = NEPI_WARPS * 32;      // epilogue threads
constexpr int WARP_MMA = NEPI_WARPS;       // issues every tcgen05.mma (one elected lane) + bulk prefetches
constexpr int WARP_LOAD = NEPI_WARPS + 1;  // builds the F-wide operand tile of the NEXT period (off the critical path)
constexpr int NTHREADS = NEPI + 64;

// Gate nonlinearities: the single-MUFU tanh.approx.f32 (max relative error 2^-11, below the bf16 operand
// rounding of 2^-9), sigmoid(v) = 0.5 tanh(v/2) + 0.5 -- the kernel is MUFU-bound otherwise.
__device__ __forceinline__ float fast_tanh(float v) {
  float r;
  asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float fast_sigmoid(float v) { return fmaf(0.5f, fast_tanh(0.5f * v), 0.5f); }

// ------------------------------------------------------------------------------------------
// weight image: fp32 collapsed weights (k_prep) -> swizzled operand tiles
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void put_w(uint8_t* tile0, bool chunk_tile, int rows, int r, int c, float v) {
  const uint32_t off = chunk_tile ? chunk_off(r, (c * 2) >> 4, rows) + ((c * 2) & 15) : sw128_off(r, c * 2, rows);
  *reinterpret_cast<__nv_bfloat16*>(tile0 + off) = __float2bfloat16(v);
}

// Wzr [F+H][2H], Wc [F+H][H] (rows 0..F-1: S part, rows F..: h part), lin_w[g] [H][2H]
template <int HH>
__global__ void k_pack_tc(const float* __restrict__ Wzr, const float* __restrict__ Wc, const float* __restrict__ czr,
                          const float* __restrict__ cc, const float* __restrict__ c0, const float* __restrict__ M0t,
                          const float* __restrict__ M1t, const float* __restrict__ probs, int T,
                          const float* __restrict__ lw0, const float* __restrict__ lw1, const float* __restrict__ lw2,
                          uint8_t* __restrict__ img_f, uint8_t* __restrict__ img_b) {
  using Cfg = TcCfg<HH>;
  constexpr int SKE = 16;  // elements of the padded S part
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  constexpr int n_zr_h = 2 * HH * HH, n_zr_s = 2 * HH * SKE, n_c_h = HH * HH, n_c_s = HH * SKE;
  int j = i;
  if (j < n_zr_h) {
    const int n = j / HH, k = j % HH;
    put_w(img_f, false, 2 * HH, n, k, Wzr[(size_t)(F + k) * 2 * HH + n]);
    return;
  }
  j -= n_zr_h;
  if (j < n_zr_s) {
    const int n = j / SKE, f = j % SKE;
    put_w(img_f + Cfg::WZR_H, true, 2 * HH, n, f, f < F ? Wzr[(size_t)f * 2 * HH + n] : 0.f);
    return;
  }
  j -= n_zr_s;
  if (j < n_c_h) {
    const int n = j / HH, k = j % HH;
    put_w(img_f + Cfg::WZR_H + Cfg::WZR_S, false, HH, n, k, Wc[(size_t)(F + k) * HH + n]);
    return;
  }
  j -= n_c_h;
  if (j < n_c_s) {
    const int n = j / SKE, f = j % SKE;
    put_w(img_f + Cfg::WZR_H + Cfg::WZR_S + Cfg::WC_H, true, HH, n, f, f < F ? Wc[(size_t)f * HH + n] : 0.f);
    return;
  }
  j -= n_c_s;
  if (j < Cfg::C_FLOATS) {
    float v = 0.f;
    if (j < Cfg::C_CC) v = czr[j];
    else if (j < Cfg::C_C0) v = cc[j - Cfg::C_CC];
    else if (j < Cfg::C_M0) v = c0 ? c0[j - Cfg::C_C0] : 0.f;
    else if (j < Cfg::C_M1) v = M0t ? M0t[j - Cfg::C_M0] : 0.f;
    else if (j < Cfg::C_PROBS) v = M1t ? M1t[j - Cfg::C_M1] : 0.f;
    else v = (j - Cfg::C_PROBS) < T ? probs[j - Cfg::C_PROBS] : 0.f;
    reinterpret_cast<float*>(img_f + Cfg::FWD_W)[j] = v;
    reinterpret_cast<float*>(img_b + Cfg::BWD_W)[j] = v;
    return;
  }
  j -= Cfg::C_FLOATS;
  if (j < 3 * HH * HH) {  // backward: Bt_g[k][n] = linear_g.weight[n][HH + k]
    const int g = j / (HH * HH), rem = j % (HH * HH);
    const int k = rem / HH, n = rem % HH;
    const float* lw = g == 0 ? lw0 : (g == 1 ? lw1 : lw2);
    put_w(img_b + g * Cfg::BT, false, HH, k, n, lw[(size_t)n * 2 * HH + HH + k]);
    return;
  }
  j -= 3 * HH * HH;
  if (j < HH * 16) {  // B0[n][k]: k < 8 -> M0[n][k], k >= 8 -> M1[0][n][k-8]   (forward and backward images)
    const int n = j / 16, k = j % 16;
    const float v = k < F ? (M0t ? M0t[k * HH + n] : 0.f) : (M1t ? M1t[(k - F) * HH + n] : 0.f);
    put_w(img_f + Cfg::OFF_W0, true, HH, n, k, v);
    put_w(img_b + 3 * Cfg::BT, true, HH, n, k, v);
  }
}

// ------------------------------------------------------------------------------------------
// shared device helpers
// ------------------------------------------------------------------------------------------
// write CW consecutive columns [c0, c0+CW) of row r into the [128 x HH] SW128 operand tile
__device__ __forceinline__ void store_operand(uint8_t* tile, int r, int c0, const float (&v)[CW]) {
#pragma unroll
  for (int j = 0; j < CW; j += 8) {
    uint4 p;
    p.x = pack_bf16(v[j], v[j + 1]);
    p.y = pack_bf16(v[j + 2], v[j + 3]);
    p.z = pack_bf16(v[j + 4], v[j + 5]);
    p.w = pack_bf16(v[j + 6], v[j + 7]);
    *reinterpret_cast<uint4*>(tile + sw128_off(r, (c0 + j) * 2, TC_ROWS)) = p;
  }
}
// write the 8 F-wide values of row r into a chunk tile (8 bf16 = one 16-byte chunk)
__device__ __forceinline__ void store_small8(uint8_t* tile, int r, int elem0, const float (&v)[8]) {
  uint4 p;
  p.x = pack_bf16(v[0], v[1]);
  p.y = pack_bf16(v[2], v[3]);
  p.z = pack_bf16(v[4], v[5]);
  p.w = pack_bf16(v[6], v[7]);
  *reinterpret_cast<uint4*>(tile + chunk_off(r, elem0 / 8, TC_ROWS)) = p;
}

// one contraction D[128 x N] = [h-part | S-part] x W
template <int HH>
__device__ __forceinline__ void issue_gate_mma(uint32_t tmem_d, uint32_t a_h, uint32_t a_s, uint32_t w_h, uint32_t w_s,
                                               int n_rows_w, uint32_t idesc) {
  uint32_t acc = 0;
#pragma unroll
  for (int s = 0; s < HH / TcCfg<HH>::UK; ++s) {
    const int kb = s * 32;
    const uint64_t da = make_desc(a_h + (kb >> 7) * TC_ROWS * 128 + (kb & 127), 16, 1024, LAYOUT_SW128);
    const uint64_t db = make_desc(w_h + (kb >> 7) * n_rows_w * 128 + (kb & 127), 16, 1024, LAYOUT_SW128);
    umma<FMT_BF16>(tmem_d, da, db, idesc, acc);
    acc = 1;
  }
  umma<FMT_BF16>(tmem_d, make_desc(a_s, TC_ROWS * 16, 128, LAYOUT_NONE), make_desc(w_s, n_rows_w * 16, 128, LAYOUT_NONE), idesc, 1);
}

// h[CW] for columns [c0, c0+CW) of row q at period t (regional combine on F-wide features)
template <int HH>
__device__ __forceinline__ void compute_h(const TcArgs& a, const float* consts_s, bool valid, long long q, int b, int s0,
                                          int s1, int t, int c0, float (&h)[CW], float (&sv)[8]) {
  using C = TcCfg<HH>;
  float xv[8];
  {
    const size_t ro = ((size_t)t * a.BN + (valid ? q : 0)) * F;
    const float4 x0 = __ldg(reinterpret_cast<const float4*>(a.Xt + ro)), x1 = __ldg(reinterpret_cast<const float4*>(a.Xt + ro) + 1);
    const float4 s0v = __ldg(reinterpret_cast<const float4*>(a.St + ro)), s1v = __ldg(reinterpret_cast<const float4*>(a.St + ro) + 1);
    const float m = valid ? 1.f : 0.f;
    xv[0] = m * x0.x; xv[1] = m * x0.y; xv[2] = m * x0.z; xv[3] = m * x0.w;
    xv[4] = m * x1.x; xv[5] = m * x1.y; xv[6] = m * x1.z; xv[7] = m * x1.w;
    sv[0] = m * s0v.x; sv[1] = m * s0v.y; sv[2] = m * s0v.z; sv[3] = m * s0v.w;
    sv[4] = m * s1v.x; sv[5] = m * s1v.y; sv[6] = m * s1v.z; sv[7] = m * s1v.w;
  }
#pragma unroll
  for (int j = 0; j < CW; ++j) h[j] = consts_s[C::C_C0 + c0 + j];
#pragma unroll
  for (int f = 0; f < F; ++f) {
#pragma unroll
    for (int j = 0; j < CW; j += 4) {
      const float4 w = *reinterpret_cast<const float4*>(consts_s + C::C_M0 + f * HH + c0 + j);
      h[j] = fmaf(xv[f], w.x, h[j]);
      h[j + 1] = fmaf(xv[f], w.y, h[j + 1]);
      h[j + 2] = fmaf(xv[f], w.z, h[j + 2]);
      h[j + 3] = fmaf(xv[f], w.w, h[j + 3]);
    }
  }
  for (int s = s0; s < s1; ++s) {
    const int reg = a.seg_reg[s];
    const float4* up = reinterpret_cast<const float4*>(a.Ut + (((size_t)t * a.Bsz + b) * a.nseg + s) * F);
    const float4 u0 = __ldg(up), u1 = __ldg(up + 1);
    const float uv[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    if (reg == 0) {
#pragma unroll
      for (int f = 0; f < F; ++f) {
#pragma unroll
        for (int j = 0; j < CW; j += 4) {
          const float4 w = *reinterpret_cast<const float4*>(consts_s + C::C_M1 + f * HH + c0 + j);
          h[j] = fmaf(uv[f], w.x, h[j]);
          h[j + 1] = fmaf(uv[f], w.y, h[j + 1]);
          h[j + 2] = fmaf(uv[f], w.z, h[j + 2]);
          h[j + 3] = fmaf(uv[f], w.w, h[j + 3]);
        }
      }
    } else {
      const float* m = a.M1t + (size_t)reg * F * HH + c0;
#pragma unroll
      for (int f = 0; f < F; ++f) {
#pragma unroll
        for (int j = 0; j < CW; j += 4) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(m + f * HH + j));
          h[j] = fmaf(uv[f], w.x, h[j]);
          h[j + 1] = fmaf(uv[f], w.y, h[j + 1]);
          h[j + 2] = fmaf(uv[f], w.z, h[j + 2]);
          h[j + 3] = fmaf(uv[f], w.w, h[j + 3]);
        }
      }
    }
  }
  if (a.mode == REGT_MODE_REGIONAL) {
#pragma unroll
    for (int j = 0; j < CW; ++j) h[j] = h[j] > 0.f ? h[j] : 0.01f * h[j];
  }
}

// Saved-plane tile layout: one (t, q-tile) tile is contiguous so the backward can bulk-copy it.
//   bf16 planes (Z, R, H~): [T][nqt][HH/8][128][8]      fp32 plane (d h_pre): [T][nqt][HH/4][128][4]
// Thread r writes 16-byte pieces; a warp instruction covers 512 contiguous bytes.
template <typename E, int HH>
struct PlaneIO {
  static constexpr bool BF = sizeof(E) == 2;
  static constexpr int TILE_BYTES = TC_ROWS * HH * (BF ? 2 : 4);
  __device__ static __forceinline__ uint8_t* tile(void* plane, int nqt, int t, int qt) {
    return reinterpret_cast<uint8_t*>(plane) + ((size_t)t * nqt + qt) * TILE_BYTES;
  }
  // 16-byte piece index of column c for row r inside a tile
  __device__ static __forceinline__ uint32_t piece_off(int r, int c) {
    return (uint32_t)(((c / (BF ? 8 : 4)) * TC_ROWS + r) * 16);
  }
  __device__ static __forceinline__ void store(void* plane, int nqt, int t, int qt, int r, int c0, const float (&v)[CW]) {
    uint8_t* tb = tile(plane, nqt, t, qt);
    if constexpr (BF) {
#pragma unroll
      for (int j = 0; j < CW; j += 8) {
        uint4 p;
        p.x = pack_bf16(v[j], v[j + 1]);
        p.y = pack_bf16(v[j + 2], v[j + 3]);
        p.z = pack_bf16(v[j + 4], v[j + 5]);
        p.w = pack_bf16(v[j + 6], v[j + 7]);
        *reinterpret_cast<uint4*>(tb + piece_off(r, c0 + j)) = p;
      }
    } else {
#pragma unroll
      for (int j = 0; j < CW; j += 4)
        *reinterpret_cast<float4*>(tb + piece_off(r, c0 + j)) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    }
  }
  // read CW columns of row r from a tile image (global or shared)
  __device__ static __forceinline__ void load(const uint8_t* tb, int r, int c0, float (&v)[CW]) {
    if constexpr (BF) {
#pragma unroll
      for (int j = 0; j < CW; j += 8) {
        const uint4 p = *reinterpret_cast<const uint4*>(tb + piece_off(r, c0 + j));
        const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          v[j + 2 * e] = __uint_as_float(w[e] << 16);
          v[j + 2 * e + 1] = __uint_as_float(w[e] & 0xFFFF0000u);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < CW; j += 4) {
        const float4 p = *reinterpret_cast<const float4*>(tb + piece_off(r, c0 + j));
        v[j] = p.x; v[j + 1] = p.y; v[j + 2] = p.z; v[j + 3] = p.w;
      }
    }
  }
};

// ------------------------------------------------------------------------------------------
// per-row F-wide features of one period (period-major arrays written by k_feat_tc)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_feats(const TcArgs& a, bool valid, long long q, int b, int s0, int s1, int t,
                                           float (&sv)[8], float (&xv)[8], float (&uv)[8]) {
  const size_t ro = ((size_t)t * a.BN + (valid ? q : 0)) * F;
  const float4 x0 = __ldg(reinterpret_cast<const float4*>(a.Xt + ro)), x1 = __ldg(reinterpret_cast<const float4*>(a.Xt + ro) + 1);
  const float4 q0 = __ldg(reinterpret_cast<const float4*>(a.St + ro)), q1 = __ldg(reinterpret_cast<const float4*>(a.St + ro) + 1);
  float4 u0 = make_float4(0.f, 0.f, 0.f, 0.f), u1 = u0;
  if (s1 > s0) {
    const float4* up = reinterpret_cast<const float4*>(a.Ut + (((size_t)t * a.Bsz + b) * a.nseg + s0) * F);
    u0 = __ldg(up);
    u1 = __ldg(up + 1);
  }
  const float m = valid ? 1.f : 0.f;
  xv[0] = m * x0.x; xv[1] = m * x0.y; xv[2] = m * x0.z; xv[3] = m * x0.w;
  xv[4] = m * x1.x; xv[5] = m * x1.y; xv[6] = m * x1.z; xv[7] = m * x1.w;
  sv[0] = m * q0.x; sv[1] = m * q0.y; sv[2] = m * q0.z; sv[3] = m * q0.w;
  sv[4] = m * q1.x; sv[5] = m * q1.y; sv[6] = m * q1.z; sv[7] = m * q1.w;
  uv[0] = u0.x; uv[1] = u0.y; uv[2] = u0.z; uv[3] = u0.w; uv[4] = u1.x; uv[5] = u1.y; uv[6] = u1.z; uv[7] = u1.w;
}

// forward small tile: S (+ zero pad) | X | U
template <int HH>
__device__ __forceinline__ void write_small_fwd(uint8_t* sm, int r, const float (&sv)[8], const float (&xv)[8],
                                                const float (&uv)[8]) {
  constexpr int XU = TcCfg<HH>::SMF_XU_CHUNK * 8;   // first element of the X | U part (8 bf16 per chunk)
  store_small8(sm, r, 0, sv);
  *reinterpret_cast<uint4*>(sm + chunk_off(r, 1, TC_ROWS)) = make_uint4(0, 0, 0, 0);
  store_small8(sm, r, XU, xv);
  store_small8(sm, r, XU + 8, uv);
}

// h_pre[128 x HH] = [X | U] x [M0 ; M1]   (K = 16: one MMA)
template <int HH>
__device__ __forceinline__ void issue_h_mma(uint32_t tmem_d, uint32_t sm_xu, uint32_t w0) {
  umma<FMT_BF16>(tmem_d, make_desc(sm_xu, TC_ROWS * 16, 128, LAYOUT_NONE), make_desc(w0, HH * 16, 128, LAYOUT_NONE),
                 make_idesc(FMT_BF16, 128, HH, 0, 0), 0);
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
// step s of a CTA -> (item, period): items blockIdx.x, +gridDim.x, ... ; tp periods per item
struct StepIt {
  int item, t, ti;
  __device__ __forceinline__ void set(const TcArgs& a, int s) {
    const int k = s / a.tp;
    ti = s - k * a.tp;
    item = blockIdx.x + k * gridDim.x;
    t = (item % a.ntc) * a.tp + ti;
  }
};
__device__ __forceinline__ int cta_steps(const TcArgs& a) {
  const int n_items = (a.items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  return n_items * a.tp;
}
__device__ __forceinline__ bool ri_valid(const TcArgs& a, int item, int r) {
  return (long long)(item / a.ntc) * TC_ROWS + r < a.BN;
}
struct RowInfo {
  long long q;
  int b, s0, s1;
  bool valid;
  __device__ __forceinline__ void set(const TcArgs& a, int item, int r, bool need_seg) {
    q = (long long)(item / a.ntc) * TC_ROWS + r;
    valid = q < a.BN;
    b = valid ? (int)(q / a.N) : 0;
    s0 = s1 = 0;
    if (valid && need_seg) {
      const int n = (int)(q - (long long)b * a.N);
      s0 = a.seg_ptr[n];
      s1 = a.seg_ptr[n + 1];
    }
  }
};

template <int HH>
__global__ void __launch_bounds__(NTHREADS, 1) k_cell_fwd_tc(TcArgs a) {
  using Cfg = TcCfg<HH>;
  using PIO = PlaneIO<__nv_bfloat16, HH>;
  constexpr int NBUF = 2;                              // small-tile buffers
  constexpr int SMB = Cfg::SMF_TILE;                   // bytes per small-tile buffer
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // align inside the shared window with pointer arithmetic only (an integer round trip would make
  // every later access a generic LD/ST instead of LDS/STS)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* W = smem;                                   // weight image (tiles + consts)
  uint8_t* Ah = W + ((Cfg::FWD_IMG + 1023) & ~1023);   // [128 x HH] operand tile: h, then h*R
  uint8_t* SMf = Ah + Cfg::A_TILE;                     // [NBUF] small tiles  S(+pad) | X | U
  __shared__ uint64_t bar_a, bar_zr, bar_a2, bar_c, bar_img, bar_h;
  __shared__ uint64_t bar_x[2];   // per small-tile buffer, like bar_free: tile written / tile consumed
  // bar_free[b]: completes once per use of small-tile buffer b (the MMAs that read it are done).  The
  // loader waits on it instead of bar_c: a waiter may lag an mbarrier by at most ONE phase, and only
  // a per-buffer barrier guarantees that (its next phase needs the loader's own next tile).
  __shared__ uint64_t bar_free[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    mbar_init(&bar_free[0], 1);
    mbar_init(&bar_free[1], 1);
    mbar_init(&bar_a, NEPI);
    mbar_init(&bar_zr, 1);
    mbar_init(&bar_a2, NEPI);
    mbar_init(&bar_c, 1);
    mbar_init(&bar_img, 1);
    mbar_init(&bar_x[0], 1);
    mbar_init(&bar_x[1], 1);
    mbar_init(&bar_h, 1);
    fence_barrier_init();
    // weight image -> shared memory with the bulk-copy engine (16 KB pieces)
    mbar_arrive_expect_tx(&bar_img, Cfg::FWD_IMG);
    for (int o = 0; o < Cfg::FWD_IMG; o += 16384)
      bulk_g2s(W + o, a.img + o, min(16384, Cfg::FWD_IMG - o), &bar_img);
  }
  if (warp == WARP_MMA) tmem_alloc(&tmem_base_s, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // the loader warp does not read the weight image: it starts on the first tile while the image lands
  if (warp != WARP_LOAD) mbar_wait(&bar_img, 0);
  const uint32_t tmem = tmem_base_s;
  const float* consts = reinterpret_cast<const float*>(W + Cfg::FWD_W);
  const bool hmma = a.hmma != 0;
  const int S = cta_steps(a);

  if (warp < NEPI_WARPS) {
    // ================= epilogue threads: thread = (row r, CW columns) =================
    const int r = (warp & 3) * 32 + lane;  // row = TMEM lane
    const int ch = warp >> 2;              // column group
    const int c0 = ch * CW;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    RowInfo ri;
    float acc[CW];
    StepIt it;
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      it.set(a, s);
      const int qt = it.item / a.ntc;
      if (it.ti == 0) {
        ri.set(a, it.item, r, !hmma);
#pragma unroll
        for (int j = 0; j < CW; ++j) acc[j] = 0.f;
      }
      float h[CW];
      if (hmma) {
        mbar_wait(&bar_h, ph);
        tc_fence_after();
        tmem_ld<CW>(tlane + 3 * HH + c0, h);
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          const float v = h[j] + consts[Cfg::C_C0 + c0 + j];
          h[j] = (a.mode == REGT_MODE_REGIONAL) ? (v > 0.f ? v : 0.01f * v) : v;
        }
      } else {
        float sv[8];
        compute_h<HH>(a, consts, ri.valid, ri.q, ri.b, ri.s0, ri.s1, it.t, c0, h, sv);
      }
      store_operand(Ah, r, c0, h);
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_a);

      // ---- E1: gates ----
      mbar_wait(&bar_zr, ph);
      tc_fence_after();
      float z[CW];
      {
        float raw[CW];
        tmem_ld<CW>(tlane + c0, raw);
#pragma unroll
        for (int j = 0; j < CW; ++j) z[j] = fast_sigmoid(raw[j] + consts[Cfg::C_CZR + c0 + j]);
        PIO::store(a.Zp, a.nqt, it.t, qt, r, c0, z);
        tmem_ld<CW>(tlane + HH + c0, raw);
        float hr[CW];
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          const float rg = fast_sigmoid(raw[j] + consts[Cfg::C_CZR + HH + c0 + j]);
          raw[j] = rg;
          hr[j] = h[j] * rg;
        }
        PIO::store(a.Rp, a.nqt, it.t, qt, r, c0, raw);
        store_operand(Ah, r, c0, hr);
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_a2);

      // ---- E2: candidate, blend, attention accumulation ----
      mbar_wait(&bar_c, ph);
      tc_fence_after();
      {
        float raw[CW];
        tmem_ld<CW>(tlane + 2 * HH + c0, raw);
        const float pt = consts[Cfg::C_PROBS + it.t];
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          const float hc = fast_tanh(raw[j] + consts[Cfg::C_CC + c0 + j]);
          raw[j] = hc;
          acc[j] = fmaf(pt, z[j] * h[j] + (1.0f - z[j]) * hc, acc[j]);
        }
        PIO::store(a.Hcp, a.nqt, it.t, qt, r, c0, raw);
      }
      if (it.ti + 1 == a.tp) {   // item done: its partial attention sum, tile layout [chunk][qt][HH/4][128][4]
        float4* o = reinterpret_cast<float4*>(a.hid_part) + ((size_t)(it.item % a.ntc) * a.nqt + qt) * (HH / 4) * TC_ROWS;
#pragma unroll
        for (int j = 0; j < CW; j += 4)
          o[(size_t)((c0 + j) >> 2) * TC_ROWS + r] = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
      }
    }
    tc_fence_before();
  } else if (warp == WARP_MMA) {
    // ================= MMA issuer (one elected lane) =================
    const uint32_t idesc_zr = make_idesc(FMT_BF16, 128, 2 * HH, 0, 0), idesc_c = make_idesc(FMT_BF16, 128, HH, 0, 0);
    const uint32_t ah = smem_u32(Ah), smf = smem_u32(SMf), w = smem_u32(W);
    constexpr int XU = Cfg::SMF_XU_CHUNK * TC_ROWS * 16;             // offset of the X | U chunks
    if (S > 0) {  // the loader has built step 0's tile: h_pre of step 0
      mbar_wait(&bar_x[0], 0);
      tc_fence_after();
      if (lane == 0 && hmma) {
        issue_h_mma<HH>(tmem + 3 * HH, smf + XU, w + Cfg::OFF_W0);
        umma_commit(&bar_h);
      }
      __syncwarp();
    }
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      const uint32_t as = smf + (s % NBUF) * SMB;
      mbar_wait(&bar_a, ph);
      tc_fence_after();
      if (lane == 0) {
        issue_gate_mma<HH>(tmem, ah, as, w, w + Cfg::WZR_H, 2 * HH, idesc_zr);
        umma_commit(&bar_zr);
      }
      __syncwarp();
      mbar_wait(&bar_a2, ph);
      tc_fence_after();
      if (lane == 0) {
        issue_gate_mma<HH>(tmem + 2 * HH, ah, as, w + Cfg::WZR_H + Cfg::WZR_S, w + Cfg::WZR_H + Cfg::WZR_S + Cfg::WC_H, HH,
                           idesc_c);
        umma_commit(&bar_c);
        umma_commit(&bar_free[s % NBUF]);
      }
      __syncwarp();
      if (s + 1 < S) {  // next period's small tile (built by the loader warp) -> its h_pre
        mbar_wait(&bar_x[(s + 1) % NBUF], (uint32_t)(((s + 1) / NBUF) & 1));
        tc_fence_after();
        if (lane == 0 && hmma) {
          issue_h_mma<HH>(tmem + 3 * HH, smf + ((s + 1) % NBUF) * SMB + XU, w + Cfg::OFF_W0);
          umma_commit(&bar_h);
        }
        __syncwarp();
      }
    }
    tc_fence_before();
  } else {
    // ================= loader warp: S(+pad) | X | U of the next period, 4 rows per lane =================
    RowInfo ri[4];
    StepIt it;
    for (int s = 0; s < S; ++s) {
      it.set(a, s);
      if (it.ti == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) ri[k].set(a, it.item, lane + 32 * k, true);
      }
      float sv[4][8], xv[4][8], uv[4][8];
#pragma unroll
      for (int k = 0; k < 4; ++k) load_feats(a, ri[k].valid, ri[k].q, ri[k].b, ri[k].s0, ri[k].s1, it.t, sv[k], xv[k], uv[k]);
      // buffer s % NBUF was last read by the MMAs of step s - NBUF: use number s / NBUF - 1 of that buffer
      if (s >= NBUF) mbar_wait(&bar_free[s % NBUF], (uint32_t)((s / NBUF - 1) & 1));
      uint8_t* sm = SMf + (s % NBUF) * SMB;
#pragma unroll
      for (int k = 0; k < 4; ++k) write_small_fwd<HH>(sm, lane + 32 * k, sv[k], xv[k], uv[k]);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_x[s % NBUF]);
    }
  }
  __syncthreads();
  if (warp == WARP_MMA) tmem_dealloc(tmem, 256);
}

// out_hidden[q][j] = sum over the t-chunks of the per-item partial attention sums (tiled partials, see above)
__global__ void k_hid_reduce(const float* __restrict__ part, int ntc, int nqt, int HH, long long BN, float* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // one float4 of out
  const int h4 = HH >> 2;
  if (i >= BN * h4) return;
  const long long q = i / h4;
  const int c4 = (int)(i - q * h4);
  const size_t tile = (size_t)h4 * TC_ROWS;   // float4 per (chunk, qt) tile
  const float4* p = reinterpret_cast<const float4*>(part) + (size_t)(q >> 7) * tile + (size_t)c4 * TC_ROWS + (q & 127);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int c = 0; c < ntc; ++c) {
    const float4 v = __ldg(p + (size_t)c * nqt * tile);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  reinterpret_cast<float4*>(out)[i] = s;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// periods per work item: maximise SM utilisation of the last wave, prefer longer chunks
static int choose_tp(int nqt, int T, int slots) {
  int best = 1;
  double best_eff = -1.0;
  for (int tp = T; tp >= 1; --tp) {
    if (T % tp) continue;
    const long long items = (long long)nqt * (T / tp);
    const long long waves = (items + slots - 1) / slots;
    const double eff = (double)items / (double)(waves * slots);
    if (eff > best_eff + 0.02) {
      best_eff = eff;
      best = tp;
    }
  }
  return best;
}

int tc_num_chunks(const regt_args* a) {
  const int BN = a->B * a->N, nqt = (BN + TC_ROWS - 1) / TC_ROWS;
  return a->T / choose_tp(nqt, a->T, sm_count());
}

static TcArgs make_tcargs(const regt_args* a, const Layout& L, int slots) {
  TcArgs k{};
  k.BN = a->B * a->N; k.N = a->N; k.T = a->T; k.nseg = a->plan.nseg; k.mode = a->mode;
  k.hmma = (a->plan.R == 1) ? 1 : 0;   // one regional list: every row uses the same M1 block
  k.nqt = (k.BN + TC_ROWS - 1) / TC_ROWS;
  k.tp = choose_tp(k.nqt, a->T, slots);
  k.ntc = a->T / k.tp;
  k.items = k.nqt * k.ntc;
  k.Xt = L.Xt; k.St = L.S; k.Ut = L.U; k.Bsz = a->B;
  k.seg_ptr = a->plan.seg_ptr; k.seg_reg = a->plan.seg_reg;
  k.M1t = L.M1t;
  k.img = L.tc_img_f;
  k.Zp = L.Zp; k.Rp = L.Rp; k.Hcp = L.Hcp; k.hid_part = L.hid_part;
  k.G = L.G; k.dhp = L.dhp_p; k.wpart = L.tc_wpart; k.dprobs_part = L.tc_dpp;
  return k;
}
// persistent grids: one CTA per SM at most; the backward's per-CTA weight-gradient partials hold TC_MAX_CTAS
static int tc_fwd_grid(const TcArgs& k, int slots) { return min(slots, k.items); }
static int tc_bwd_grid(const TcArgs& k, int slots) { return min(tc_fwd_grid(k, slots), TC_MAX_CTAS); }

template <int HH>
static int run_fwd_tc(const regt_args* a, const Layout& L, cudaStream_t st, bool forked) {
  using Cfg = TcCfg<HH>;
  static_assert(Cfg::FWD_IMG <= TC_IMG_BYTES && Cfg::BWD_IMG <= TC_IMG_BYTES, "weight image too large");
  const int n_pack = 2 * HH * HH + 2 * HH * 16 + HH * HH + HH * 16 + Cfg::C_FLOATS + 3 * HH * HH + HH * 16;
  k_pack_tc<HH><<<cdiv(n_pack, 256), 256, 0, st>>>(L.Wzr, L.Wc, L.czr, L.cc, L.c0, L.M0t, L.M1t, L.probs, a->T,
                                                  a->p.lin_w[0], a->p.lin_w[1], a->p.lin_w[2], L.tc_img_f, L.tc_img_b);
  REGT_LAUNCHED("k_pack_tc", st);
  if (forked && join_side(st)) return -1;   // the feature builder ran beside the weight collapse
  const int slots = sm_count();
  TcArgs k = make_tcargs(a, L, slots);
  const size_t smem = 1024 + ((Cfg::FWD_IMG + 1023) & ~1023) + Cfg::A_TILE + 2 * Cfg::SMF_TILE;
  REGT_CUDA(cudaFuncSetAttribute(k_cell_fwd_tc<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = tc_fwd_grid(k, slots);
  k_cell_fwd_tc<HH><<<grid, NTHREADS, smem, st>>>(k);
  REGT_LAUNCHED("k_cell_fwd_tc", st);
  if (!L.route.hid_partials) {  // otherwise the head sums the partials while loading its tiles
    const long long count = (long long)k.BN * HH;
    k_hid_reduce<<<cdiv(count / 4, 256), 256, 0, st>>>(L.hid_part, k.ntc, k.nqt, HH, k.BN, a->out_hidden);
    REGT_LAUNCHED("k_hid_reduce", st);
  }
  return 0;
}

bool cell_tc_fits(const regt_args* a) { return a->H == 64 && a->mode != REGT_MODE_TGCN; }

int cell_forward_tc(const regt_args* a, const Layout& L, cudaStream_t st) {
  REGT_CHECK(a->H == 64, "the fused bf16 tensor-core kernels are built for hidden=64 (got %d); use precision tf32x3 or fp32", a->H);
  REGT_CHECK(a->mode != REGT_MODE_TGCN, "tensor-core precisions do not cover the bare TGCN cell; use precision fp32");
  REGT_CHECK(a->T <= 64, "tensor-core path supports up to 64 periods");
  // features (graph + x) and collapsed weights (parameters) are independent: two streams
  cudaStream_t side = fork_side(st);
  if (launch_feat_tc(a->plan, a->x, feat_in(a), a->B, a->x_rows > 0 ? a->x_rows : a->N, a->T, L.Xt, L.S, L.U, side ? side : st)) return -1;
  if (launch_prep(a, L, st)) return -1;
  return run_fwd_tc<64>(a, L, st, side != nullptr);
}

// ------------------------------------------------------------------------------------------
// backward (bf16 operands): data gradients and ALL weight gradients on the tensor cores
// ------------------------------------------------------------------------------------------
// Per period and 128-row tile (same work items / thread ownership as the forward):
//   H0  h_pre = [X|U] . [M0;M1]  (recompute, TMEM cols 320..383; issued one period ahead)
//   E0  h = act(h_pre + c0); read saved Z,R,H~ (bulk-prefetched tile); dH' = probs[t] G;
//       Dh = dH~ (1-H~^2), Dz = dZ Z(1-Z); operand tiles Dh, Dz, h, h*R -> smem
//   M1  dHR = Dh . B_h                                  (TMEM cols   0.. 63)
//   E1  dh += dHR R ; Dr = dHR h R(1-R) -> smem
//   M2  dhg = Dz . B_z + Dr . B_r                       (TMEM cols  64..127)
//   W1  [Dz|Dr]^T . h        -> dB_z, dB_r              (TMEM cols 128..191, persistent)
//   W1s [Dz|Dr]^T . [S|X|U|1] -> dP_z, dP_r, dc_z, dc_r (TMEM cols 192..223, persistent)
//   E2  d h_pre = act'(h) (dh + dhg) -> smem
//   W2  [Dh|dhp]^T . (h*R)   -> dB_h                    (TMEM cols 224..287, persistent)
//   W2s [Dh|dhp]^T . [S|X|U|1] -> dP_h, dc_h, dM0, dM1, dc0 (TMEM cols 288..319, persistent)
// The weight-gradient MMAs read the SAME shared-memory tiles as MN-major operands (contraction over
// the 128 rows); their accumulators live in TMEM for the whole kernel and are flushed once per CTA.
constexpr int WP_COLS = 192;  // per-CTA partial: [128][192] = accW1 | accW1s | accW2 | accW2s

template <int HH>
__global__ void __launch_bounds__(NTHREADS, 1) k_cell_bwd_tc(TcArgs a) {
  constexpr int FMT = FMT_BF16;
  using Cfg = TcCfg<HH>;
  using PIO = PlaneIO<__nv_bfloat16, HH>;
  constexpr int TILE = Cfg::A_TILE;          // 16 KB
  constexpr int PT = PIO::TILE_BYTES;        // 16 KB
  constexpr int SMT = 4 * TC_ROWS * 16;      // small tile: S | X | U | ones
  constexpr int GT = TC_ROWS * HH * 4;       // G tile (fp32, [HH/4][128][4])
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* W = smem;                                     // Bt_z | Bt_r | Bt_h | B0 | consts
  uint8_t* T_DH = W + ((Cfg::BWD_IMG + 1023) & ~1023);
  uint8_t* T_DHP = T_DH + TILE;
  uint8_t* T_DZ = T_DHP + TILE;
  uint8_t* T_DR = T_DZ + TILE;
  uint8_t* T_H = T_DR + TILE;
  uint8_t* T_HR = T_H + TILE;
  uint8_t* SM = T_HR + TILE;                             // [2] small tiles (double-buffered)
  uint8_t* STG = SM + 2 * SMT;                           // staged Z | R | H~ tiles
  uint8_t* GS = STG + 3 * PT;                            // G tile of the current item
  __shared__ uint64_t bar_stage, bar_g, bar_e0, bar_m1, bar_e1, bar_m2, bar_e2, bar_w, bar_img, bar_h;
  // per small-tile buffer: tile written by the loader / tile consumed by the MMAs.  Per-buffer barriers keep
  // every waiter within one phase of its barrier (a waiter two phases behind would block forever).
  __shared__ uint64_t bar_x[2], bar_sfree[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    mbar_init(&bar_img, 1);
    mbar_init(&bar_stage, 1);
    mbar_init(&bar_g, 1);
    mbar_init(&bar_e0, NEPI);
    mbar_init(&bar_m1, 1);
    mbar_init(&bar_e1, NEPI);
    mbar_init(&bar_m2, 1);
    mbar_init(&bar_e2, NEPI);
    mbar_init(&bar_w, 1);
    mbar_init(&bar_x[0], 1);
    mbar_init(&bar_x[1], 1);
    mbar_init(&bar_sfree[0], 1);
    mbar_init(&bar_sfree[1], 1);
    mbar_init(&bar_h, 1);
    fence_barrier_init();
    mbar_arrive_expect_tx(&bar_img, Cfg::BWD_IMG);
    for (int o = 0; o < Cfg::BWD_IMG; o += 16384)
      bulk_g2s(W + o, a.img + o, min(16384, Cfg::BWD_IMG - o), &bar_img);
  }
  if (warp == WARP_MMA) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp != WARP_LOAD) mbar_wait(&bar_img, 0);   // the loader warp does not read the weight image
  const uint32_t tmem = tmem_base_s;
  const float* consts = reinterpret_cast<const float*>(W + Cfg::BWD_W);
  const bool hmma = a.hmma != 0;
  const int S = cta_steps(a);

  if (warp < NEPI_WARPS) {
    const int r = (warp & 3) * 32 + lane;
    const int ch = warp >> 2;
    const int c0 = ch * CW;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    RowInfo ri;
    StepIt it;
    float dpr0 = 0.f, dpr1 = 0.f;   // attention-gradient sums of periods lane and 32 + lane
    // h of one step (recomputed, not saved): tensor-core h_pre (single regional list) or CUDA cores
    auto make_h = [&](const StepIt& st_, uint32_t ph_, float (&h_)[CW]) {
      if (hmma) {
        mbar_wait(&bar_h, ph_);
        tc_fence_after();
        tmem_ld<CW>(tlane + 320 + c0, h_);
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          const float v = h_[j] + consts[Cfg::C_C0 + c0 + j];
          h_[j] = (a.mode == REGT_MODE_REGIONAL) ? (v > 0.f ? v : 0.01f * v) : v;
        }
      } else {
        float sv[8];
        compute_h<HH>(a, consts, ri.valid, ri.q, ri.b, ri.s0, ri.s1, st_.t, c0, h_, sv);
      }
    };
    if (S > 0) {
      it.set(a, 0);
      ri.set(a, it.item, r, !hmma);
    }
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      it.set(a, s);
      const int qt = it.item / a.ntc;
      float h[CW], dh[CW], rr[CW];
      if (it.ti == 0 && s > 0) ri.set(a, it.item, r, !hmma);
      make_h(it, ph, h);
      const bool row_valid = ri.valid;   // ri moves on to the next item before this step ends
      if (it.ti == 0) mbar_wait(&bar_g, (uint32_t)((s / a.tp) & 1));   // this item's G tile has landed in smem
      const float pt = consts[Cfg::C_PROBS + it.t];
      float dp = 0.f;
      mbar_wait(&bar_stage, ph);
      {
        float z[CW], hc[CW];
        PIO::load(STG, r, c0, z);
        PIO::load(STG + PT, r, c0, rr);
        PIO::load(STG + 2 * PT, r, c0, hc);
#pragma unroll
        for (int j = 0; j < CW; j += 4) {
          float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);   // rows past B*N: the padded part of G is never written
          if (row_valid) g4 = reinterpret_cast<const float4*>(GS)[((c0 + j) / 4) * TC_ROWS + r];
          const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int jj = j + e;
            const float zz = z[jj], hcc = hc[jj], hv = h[jj];
            dp = fmaf(gv[e], zz * hv + (1.0f - zz) * hcc, dp);
            const float gs = pt * gv[e];
            dh[jj] = gs * zz;
            z[jj] = gs * (hv - hcc) * zz * (1.0f - zz);          // Dz
            hc[jj] = gs * (1.0f - zz) * (1.0f - hcc * hcc);      // Dh
          }
        }
        if (s > 0) mbar_wait(&bar_w, (uint32_t)((s - 1) & 1));  // previous step's MMAs released the tiles
        store_operand(T_DH, r, c0, hc);
        fence_proxy_async();
        tc_fence_before();
        mbar_arrive(&bar_e0);          // M1 needs Dh only: it runs under the remaining tile stores (62.7 against 65.5 us)
        store_operand(T_DZ, r, c0, z);
#pragma unroll
        for (int j = 0; j < CW; ++j) z[j] = h[j] * rr[j];
        store_operand(T_HR, r, c0, z);
        store_operand(T_H, r, c0, h);   // made visible to the tensor core by the fence before bar_e1
      }

      // ---- E1 ----
      mbar_wait(&bar_m1, ph);
      tc_fence_after();
      {
        float raw[CW];
        tmem_ld<CW>(tlane + c0, raw);
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          const float dHR = raw[j];
          dh[j] = fmaf(dHR, rr[j], dh[j]);
          raw[j] = dHR * h[j] * rr[j] * (1.0f - rr[j]);   // Dr
        }
        store_operand(T_DR, r, c0, raw);
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_e1);

      // ---- E2 ----
      mbar_wait(&bar_m2, ph);
      tc_fence_after();
      {
        float raw[CW];
        tmem_ld<CW>(tlane + 64 + c0, raw);
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          float v = dh[j] + raw[j];
          if (a.mode == REGT_MODE_REGIONAL) v *= (h[j] > 0.f ? 1.0f : 0.01f);
          raw[j] = v;
        }
        store_operand(T_DHP, r, c0, raw);
        if (a.mode == REGT_MODE_REGIONAL && !hmma) PlaneIO<float, HH>::store(a.dhp, a.nqt, it.t, qt, r, c0, raw);
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_e2);

      // ---- attention gradient partial: fixed-order block reduction ----
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) dp += __shfl_xor_sync(0xffffffffu, dp, d);
      // per-warp running sum of period t lives in a register of lane t % 32 (fixed order, no block
      // barrier per step); combined once per CTA after the loop
      if (lane == (it.t & 31)) {
        if (it.t < 32) dpr0 += dp;
        else dpr1 += dp;
      }
    }
    // ---- attention-gradient partial of this CTA: fixed-order sum over the epilogue warps ----
    {
      float* dpacc = reinterpret_cast<float*>(STG);   // the plane staging area is free: every prefetch was consumed
      dpacc[warp * 64 + lane] = dpr0;
      dpacc[warp * 64 + 32 + lane] = dpr1;
      asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory");
      if (tid < a.T) {
        float sacc = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < NEPI_WARPS; ++w8) sacc += dpacc[w8 * 64 + tid];
        a.dprobs_part[(size_t)blockIdx.x * a.T + tid] = sacc;
      }
    }
    // ---- flush the persistent weight-gradient accumulators ----
    mbar_wait(&bar_w, (uint32_t)((S - 1) & 1));
    tc_fence_after();
    float* wp = a.wpart + ((size_t)blockIdx.x * TC_ROWS + r) * WP_COLS;
    {
      float v[CW];
      tmem_ld<CW>(tlane + 128 + c0, v);
#pragma unroll
      for (int j = 0; j < CW; j += 4) *reinterpret_cast<float4*>(wp + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      tmem_ld<CW>(tlane + 224 + c0, v);
#pragma unroll
      for (int j = 0; j < CW; j += 4) *reinterpret_cast<float4*>(wp + 96 + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      constexpr int SW = 32 / (64 / CW);  // columns of the 32-wide accumulators per thread
      float u[SW];
      tmem_ld<SW>(tlane + 192 + ch * SW, u);
#pragma unroll
      for (int j = 0; j < SW; j += 4) *reinterpret_cast<float4*>(wp + 64 + ch * SW + j) = make_float4(u[j], u[j + 1], u[j + 2], u[j + 3]);
      tmem_ld<SW>(tlane + 288 + ch * SW, u);
#pragma unroll
      for (int j = 0; j < SW; j += 4) *reinterpret_cast<float4*>(wp + 160 + ch * SW + j) = make_float4(u[j], u[j + 1], u[j + 2], u[j + 3]);
    }
    tc_fence_before();
  } else if (warp == WARP_MMA) {
    // ================= MMA issuer + bulk prefetch of the saved planes / G tile =================
    const uint32_t id_dg = make_idesc(FMT, 128, HH, 0, 0);        // data gradients (K-major)
    const uint32_t id_w = make_idesc(FMT, 128, HH, 1, 1);         // weight gradients (MN-major)
    const uint32_t id_ws = make_idesc(FMT, 128, 32, 1, 1);
    const uint32_t w = smem_u32(W), tdh = smem_u32(T_DH), tdz = smem_u32(T_DZ), tdr = smem_u32(T_DR), th = smem_u32(T_H),
                   thr = smem_u32(T_HR), sm0 = smem_u32(SM);
    constexpr int XU = 1 * TC_ROWS * 16;  // X | U are chunks 1,2 of the small tile
    auto prefetch = [&](const StepIt& n) {
      const int qt = n.item / a.ntc;
      mbar_arrive_expect_tx(&bar_stage, 3 * PT);
      bulk_g2s(STG, PIO::tile(a.Zp, a.nqt, n.t, qt), PT, &bar_stage);
      bulk_g2s(STG + PT, PIO::tile(a.Rp, a.nqt, n.t, qt), PT, &bar_stage);
      bulk_g2s(STG + 2 * PT, PIO::tile(a.Hcp, a.nqt, n.t, qt), PT, &bar_stage);
    };
    auto fetch_g = [&](int item) {
      mbar_arrive_expect_tx(&bar_g, GT);
      bulk_g2s(GS, reinterpret_cast<const uint8_t*>(a.G) + (size_t)(item / a.ntc) * GT, GT, &bar_g);
    };
    StepIt it, nx;
    if (S > 0) {
      it.set(a, 0);
      if (lane == 0) {
        prefetch(it);
        fetch_g(it.item);
      }
      mbar_wait(&bar_x[0], 0);
      tc_fence_after();
      if (lane == 0 && hmma) {
        issue_h_mma<HH>(tmem + 320, sm0 + XU, w + 3 * Cfg::BT);
        umma_commit(&bar_h);
      }
      __syncwarp();
    }
    for (int s = 0; s < S; ++s) {
      const uint32_t ph = s & 1;
      const uint32_t accw = s > 0 ? 1u : 0u;
      const uint32_t sm = sm0 + (s & 1) * SMT;
      it.set(a, s);
      const bool more = s + 1 < S;
      if (more) nx.set(a, s + 1);
      mbar_wait(&bar_e0, ph);
      tc_fence_after();
      if (lane == 0) {
        // M1: dHR = Dh . B_h
#pragma unroll
        for (int k = 0; k < HH / 16; ++k)
          umma<FMT>(tmem, make_desc(tdh + k * 32, 16, 1024, LAYOUT_SW128),
                    make_desc(w + 2 * Cfg::BT + k * 32, 16, 1024, LAYOUT_SW128), id_dg, k > 0 ? 1u : 0u);
        umma_commit(&bar_m1);
        // this step's staged planes (and, on its last period, the item's G tile) are consumed
        if (more) {
          prefetch(nx);
          if (nx.ti == 0) fetch_g(nx.item);
        }
      }
      __syncwarp();
      if (more) {  // next period's h_pre from the tile the loader warp has built (read by the epilogue under M2)
        mbar_wait(&bar_x[(s + 1) & 1], (uint32_t)(((s + 1) >> 1) & 1));
        tc_fence_after();
        if (lane == 0 && hmma) {
          issue_h_mma<HH>(tmem + 320, sm0 + ((s + 1) & 1) * SMT + XU, w + 3 * Cfg::BT);
          umma_commit(&bar_h);
        }
        __syncwarp();
      }
      mbar_wait(&bar_e1, ph);
      tc_fence_after();
      if (lane == 0) {
        // M2: dhg = Dz . B_z + Dr . B_r
#pragma unroll
        for (int k = 0; k < HH / 16; ++k)
          umma<FMT>(tmem + 64, make_desc(tdz + k * 32, 16, 1024, LAYOUT_SW128),
                    make_desc(w + k * 32, 16, 1024, LAYOUT_SW128), id_dg, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < HH / 16; ++k)
          umma<FMT>(tmem + 64, make_desc(tdr + k * 32, 16, 1024, LAYOUT_SW128),
                    make_desc(w + Cfg::BT + k * 32, 16, 1024, LAYOUT_SW128), id_dg, 1u);
        umma_commit(&bar_m2);
      }
      __syncwarp();
      if (lane == 0) {
        // W1 / W1s: [Dz|Dr]^T . h , [Dz|Dr]^T . [S|X|U|1]   (contraction over the 128 rows)
#pragma unroll
        for (int k = 0; k < TC_ROWS / 16; ++k) {
          const uint64_t da = make_desc(tdz + k * 2048, TILE, 1024, LAYOUT_SW128);
          umma<FMT>(tmem + 128, da, make_desc(th + k * 2048, TILE, 1024, LAYOUT_SW128), id_w, (k > 0) ? 1u : accw);
          umma<FMT>(tmem + 192, da, make_desc(sm + k * 256, 128, TC_ROWS * 16, LAYOUT_NONE), id_ws, (k > 0) ? 1u : accw);
        }
      }
      __syncwarp();
      mbar_wait(&bar_e2, ph);
      tc_fence_after();
      if (lane == 0) {
        // W2 / W2s: [Dh|dhp]^T . (h*R) , [Dh|dhp]^T . [S|X|U|1]
#pragma unroll
        for (int k = 0; k < TC_ROWS / 16; ++k) {
          const uint64_t da = make_desc(tdh + k * 2048, TILE, 1024, LAYOUT_SW128);
          umma<FMT>(tmem + 224, da, make_desc(thr + k * 2048, TILE, 1024, LAYOUT_SW128), id_w, (k > 0) ? 1u : accw);
          umma<FMT>(tmem + 288, da, make_desc(sm + k * 256, 128, TC_ROWS * 16, LAYOUT_NONE), id_ws, (k > 0) ? 1u : accw);
        }
        umma_commit(&bar_w);
        umma_commit(&bar_sfree[s & 1]);
      }
      __syncwarp();
    }
    tc_fence_before();
  } else {
    // ================= loader warp: S | X | U | 1 of the next period, 4 rows per lane =================
    RowInfo ri[4];
    StepIt it;
    for (int s = 0; s < S; ++s) {
      it.set(a, s);
      if (it.ti == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) ri[k].set(a, it.item, lane + 32 * k, true);
      }
      float sv[4][8], xv[4][8], uv[4][8];
#pragma unroll
      for (int k = 0; k < 4; ++k) load_feats(a, ri[k].valid, ri[k].q, ri[k].b, ri[k].s0, ri[k].s1, it.t, sv[k], xv[k], uv[k]);
      if (s >= 2) mbar_wait(&bar_sfree[s & 1], (uint32_t)(((s >> 1) - 1) & 1));   // W1s / W2s of step s-2 were the last readers
      uint8_t* sm = SM + (s & 1) * SMT;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int row = lane + 32 * k;
        store_small8(sm, row, 0, sv[k]);
        store_small8(sm, row, 8, xv[k]);
        store_small8(sm, row, 16, uv[k]);
        *reinterpret_cast<uint4*>(sm + chunk_off(row, 3, TC_ROWS)) = make_uint4(0x00003F80u, 0, 0, 0);  // bf16 1.0
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_x[s & 1]);
    }
  }
  __syncthreads();
  if (warp == WARP_MMA) tmem_dealloc(tmem, 512);
}

// sum the per-CTA partials and scatter them into the collapsed-weight gradient buffers
__global__ void __launch_bounds__(256) k_tc_wreduce(const float* __restrict__ wpart, int ncta, int HH, int R,
                                                    float* __restrict__ dB, float* __restrict__ dP,
                                                    float* __restrict__ dcg, float* __restrict__ dM0,
                                                    float* __restrict__ dM1, float* __restrict__ dc0,
                                                    const float* __restrict__ dpp, int nqt, int T,
                                                    float* __restrict__ dprobs) {
  __shared__ float red[8][32];
  const int i = blockIdx.x * 32 + threadIdx.x;
  constexpr int NW = TC_ROWS * WP_COLS;
  // outputs [0, NW): weight-gradient partials of the CTAs; [NW, NW+T): dprobs[t] = sum_qt dpp[qt][t]
  const bool is_w = i < NW, is_p = !is_w && (i - NW) < T;
  const float s = sum_parts_32x8(is_w ? wpart : dpp, is_w ? (size_t)NW : (size_t)T, is_w ? ncta : nqt,
                                 is_w ? i : i - NW, is_w || is_p, red);
  if (threadIdx.y != 0) return;
  if (is_p) {
    dprobs[i - NW] = s;
    return;
  }
  if (!is_w) return;
  const int m = i / WP_COLS, c = i % WP_COLS;
  const int g = m / HH, n = m % HH;
  if (c < 64) {
    dB[((size_t)g * HH + n) * HH + c] = s;                     // dB_z / dB_r
  } else if (c < 96) {
    const int cc = c - 64;
    if (cc < F) dP[((size_t)g * HH + n) * F + cc] = s;
    else if (cc == 24) dcg[g * HH + n] = s;
  } else if (c < 160) {
    if (m < HH) dB[((size_t)2 * HH + m) * HH + (c - 96)] = s;  // dB_h
  } else {
    const int cc = c - 160;
    if (m < HH) {
      if (cc < F) dP[((size_t)2 * HH + m) * F + cc] = s;
      else if (cc == 24) dcg[2 * HH + m] = s;
    } else {
      if (cc >= 8 && cc < 16) dM0[(size_t)n * F + cc - 8] = s;
      else if (cc >= 16 && cc < 24) { if (R == 1) dM1[(size_t)n * F + cc - 16] = s; }
      else if (cc == 24) dc0[n] = s;
    }
  }
}

// regional decomposition (R > 1): dM1[r] from the saved d h_pre plane, one CTA per (region, z-split)
template <int HH>
__global__ void __launch_bounds__(HH) k_wgrad_m1_tc(const float* __restrict__ dhp, const float* __restrict__ U,
                                                    const int32_t* __restrict__ rseg_ptr,
                                                    const int32_t* __restrict__ rseg_list,
                                                    const int32_t* __restrict__ seg_node, int B, int N, int T, int R,
                                                    int nseg, int nqt, float* __restrict__ part) {
  const int r = blockIdx.x, n = threadIdx.x;
  const int s0 = rseg_ptr[r];
  const long long items = (long long)(rseg_ptr[r + 1] - s0) * B;
  const long long per = (items + gridDim.z - 1) / gridDim.z;
  const long long i0 = blockIdx.z * per, i1 = min(items, i0 + per);
  float acc[F];
#pragma unroll
  for (int f = 0; f < F; ++f) acc[f] = 0.f;
  for (long long i = i0; i < i1; ++i) {
    const int s = rseg_list[s0 + (int)(i / B)];
    const int b = (int)(i % B);
    const long long q = (long long)b * N + seg_node[s];
    const int qt = (int)(q / TC_ROWS), row = (int)(q % TC_ROWS);
    for (int t = 0; t < T; ++t) {
      const float d = __ldg(dhp + ((((size_t)t * nqt + qt) * (HH / 4) + n / 4) * TC_ROWS + row) * 4 + (n & 3));
      const float4* up = reinterpret_cast<const float4*>(U + (((size_t)t * B + b) * nseg + s) * F);  // period-major Ut
      const float4 u0 = __ldg(up), u1 = __ldg(up + 1);
      acc[0] = fmaf(d, u0.x, acc[0]); acc[1] = fmaf(d, u0.y, acc[1]); acc[2] = fmaf(d, u0.z, acc[2]); acc[3] = fmaf(d, u0.w, acc[3]);
      acc[4] = fmaf(d, u1.x, acc[4]); acc[5] = fmaf(d, u1.y, acc[5]); acc[6] = fmaf(d, u1.z, acc[6]); acc[7] = fmaf(d, u1.w, acc[7]);
    }
  }
  float* o = part + (((size_t)blockIdx.z * R + r) * HH + n) * F;
#pragma unroll
  for (int f = 0; f < F; ++f) o[f] = acc[f];
}

int cell_backward_tc(const regt_args* a, const Layout& L, cudaStream_t st) {
  REGT_CHECK(a->precision == REGT_PREC_BF16,
             "the tensor-core cell backward is built for precision bf16 only");
  REGT_CHECK(a->H == 64 && a->mode != REGT_MODE_TGCN, "tensor-core backward: hidden=64, TemporalGCN / RegionalTemporalGCN only");
  constexpr int HH = 64;
  using Cfg = TcCfg<HH>;
  const int slots = sm_count();
  TcArgs k = make_tcargs(a, L, slots);
  k.img = L.tc_img_b;
  const int grid = tc_bwd_grid(k, slots);
  const size_t smem = 1024 + ((Cfg::BWD_IMG + 1023) & ~1023) + 6 * Cfg::A_TILE + 2 * 4 * TC_ROWS * 16 +
                      3 * PlaneIO<__nv_bfloat16, HH>::TILE_BYTES + TC_ROWS * HH * 4;
  REGT_CUDA(cudaFuncSetAttribute(k_cell_bwd_tc<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // the head's partial sums (left by the tensor-core head in regt_head_forward) are reduced beside the cell backward
  const bool head_sum = L.route.head == HeadPath::Bf16;
  cudaStream_t side = head_sum ? fork_side(st) : nullptr;
  if (head_sum && launch_head_grad_reduce(a, L, side ? side : st)) return -1;
  k_cell_bwd_tc<HH><<<grid, NTHREADS, smem, st>>>(k);
  REGT_LAUNCHED("k_cell_bwd_tc", st);
  if (side && join_side(st)) return -1;
  const int R = a->plan.R;
  k_tc_wreduce<<<cdiv(TC_ROWS * WP_COLS + a->T, 32), dim3(32, 8), 0, st>>>(L.tc_wpart, grid, HH, R, L.dB, L.dP, L.dcg, L.dM0, L.dM1,
                                                                     L.dc0, L.tc_dpp, grid, a->T, L.dprobs);
  REGT_LAUNCHED("k_tc_wreduce", st);
  if (a->mode == REGT_MODE_REGIONAL && R > 1) {
    const int zs = (int)max(1ll, min(64ll, 1024ll / R));
    k_wgrad_m1_tc<HH><<<dim3(R, 1, zs), HH, 0, st>>>(L.dhp_p, L.U, a->plan.rseg_ptr, a->plan.rseg_list, a->plan.seg_node,
                                                    a->B, a->N, a->T, R, a->plan.nseg, k.nqt, L.part);
    REGT_LAUNCHED("k_wgrad_m1_tc", st);
    if (launch_reduce_splits(L.part, L.dM1, (long long)R * HH * F, zs, 0, st)) return -1;
  }
  return launch_chain(a, L, st);
}

}  // namespace regt

// TEST HOOK: the work split the bf16 kernels use for B snapshots of N nodes over T periods, from the code that launches
// them: out = {nqt, tp, ntc, items, forward grid, backward grid, k_head_tc grid}
extern "C" int regt_debug_tc_split(int32_t B, int32_t N, int32_t T, int32_t* out) {
  REGT_CHECK(B > 0 && N > 0 && T > 0 && out, "regt_debug_tc_split: B, N, T must be positive and out non-NULL");
  regt_args a{};
  a.B = B; a.N = N; a.T = T;
  const int slots = regt::sm_count();
  const regt::TcArgs k = regt::make_tcargs(&a, regt::Layout{}, slots);
  const int32_t v[7] = {k.nqt, k.tp, k.ntc, k.items, regt::tc_fwd_grid(k, slots), regt::tc_bwd_grid(k, slots),
                        regt::head_tc_grid(&a)};
  for (int i = 0; i < 7; ++i) out[i] = v[i];
  return 0;
}
