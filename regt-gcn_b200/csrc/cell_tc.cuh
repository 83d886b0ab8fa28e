// Shared declarations of the tcgen05 (tensor-core) cell kernels.
#pragma once
#include "common.cuh"
#include "tc_common.cuh"

namespace regt {

constexpr int TC_ROWS = 128;  // rows (b,n) per tile = UMMA M = TMEM lanes

// Byte layout of the per-step weight image (built by k_pack_tc, copied verbatim to shared memory): bf16 operand tiles.
template <int HH>
struct TcCfg {
  static constexpr int ES = 2;                                     // operand element size (bf16)
  static constexpr int UK = 16;                                    // K per MMA
  static constexpr int KBYTES = HH * ES;                          // bytes along K of the H-wide part
  static constexpr int A_TILE = TC_ROWS * KBYTES;                 // one [128 x HH] SW128 tile
  // forward weights (B operands, K-major): rows = output features
  static constexpr int WZR_H = 2 * HH * KBYTES;
  static constexpr int WZR_S = 2 * (2 * HH) * 16;
  static constexpr int WC_H = HH * KBYTES;
  static constexpr int WC_S = 2 * HH * 16;
  // regional combine on the tensor core: B0[n][k] = (M0 | M1[0]) (K = 16 = X | U), chunk tile of HH rows
  static constexpr int W0 = 2 * HH * 16;
  static constexpr int OFF_W0 = WZR_H + WZR_S + WC_H + WC_S;
  static constexpr int FWD_W = OFF_W0 + W0;                       // all parts multiples of 1024
  // small per-row operand tile of the forward ([chunk][row][16 B]): S (+pad) | X | U, double-buffered
  static constexpr int SMF_TILE = 4 * TC_ROWS * 16;
  static constexpr int SMF_XU_CHUNK = 2;                           // first chunk of the X | U part
  // fp32 constants after the tiles
  static constexpr int C_CZR = 0, C_CC = 2 * HH, C_C0 = 3 * HH, C_M0 = 4 * HH, C_M1 = 4 * HH + 8 * HH,
                       C_PROBS = 4 * HH + 16 * HH, C_FLOATS = 4 * HH + 16 * HH + 64;
  static constexpr int FWD_IMG = FWD_W + C_FLOATS * 4;
  // backward weights (B operands of the data gradients, K-major over the gate index n):
  //   Bt_g[k][n] = linear_g.weight[n][HH + k]      rows = k (hidden input index), K = n
  static constexpr int BT = HH * KBYTES;
  static constexpr int BWD_W = 3 * BT + W0;
  static constexpr int BWD_IMG = BWD_W + C_FLOATS * 4;
  static_assert(KBYTES % 128 == 0, "H-wide operand must be whole 128-byte swizzle blocks");
};

struct TcArgs {
  int BN, N, T, nseg, mode, tp, ntc, nqt, items;
  int hmma;                // 1: h_pre = [X|U] x [M0;M1] on the tensor core (single regional list)
  const float *Xt, *St, *Ut;   // period-major F-wide features [T][rows][F]
  int Bsz;
  const int32_t *seg_ptr, *seg_reg;
  const float* M1t;        // [R][F][H] fp32 (global; region 0 is also in the image)
  const uint8_t* img;      // weight image
  float *Zp, *Rp, *Hcp;    // saved planes, tile layout [T][nqt][H/4][128][4]
  float* hid_part;         // [ntc][nqt][H/4][128][4] per-chunk partial attention sums (tiled like G)
  // backward
  const float* G;          // [BN][H]
  float* dhp;              // d h_pre plane [T][nqt][H/4][128][4] (regional wgrad of M1)
  float* wpart;            // [grid][...] per-CTA weight-gradient partials
  float* dprobs_part;      // [grid][T]
};

}  // namespace regt
