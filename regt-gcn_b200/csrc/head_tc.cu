// tcgen05 (sm_100a tensor core) fused training head, bf16 operands / fp32 accumulate (REGT_PREC_BF16).
//
// Replaces, for one 128-row tile of (b,n) rows at a time, the decoder MLP of the reference
// (models/RegionalTemporalGCN.py:35-38, models/TemporalGCN.py:28-31), the MSE loss of the call site
// (run.py:180) and the autograd of both (run.py:190):
//   P0  CUDA cores : hid = sum of the cell's per-chunk attention partials -> out_hidden; relu(hid) -> A0 tile
//   M1  tcgen05.mma: a1_pre[128x128] = A0[128x64] . W1^T
//   P1  CUDA cores : a1 = relu(a1_pre + b1) -> A1 tile
//   M2  tcgen05.mma: out[128x16] = A1[128x128] . W2^T                       (O <= 16, zero padded)
//   P2  CUDA cores : out += b2 -> out; diff = out - y; loss; d_out = 2 diff / (N O) -> Do tile
//                    (or the MAE / a masked mean: LossX, common.cuh, with a scale per row: a tile may span two snapshots)
//   M3  tcgen05.mma: da1_pre[128x128] = Do[128x16] . W2     ;  dW2^T[128x16] += A1^T . Do   (over rows)
//   P3  CUDA cores : d a1 = da1_pre * (a1 > 0) -> D1 tile
//   M4  tcgen05.mma: G_pre[128x64] = D1[128x128] . W1       ;  dW1[128x64] += D1^T . A0 ; db1 += D1^T . 1
//   P4  CUDA cores : G = G_pre * (hid > 0) (+ d_hidden) -> G tiles for the cell backward
// The weight-gradient MMAs read the SAME shared-memory tiles as MN-major operands (contraction over
// the tile's 128 rows); their accumulators stay in TMEM for the whole kernel and are flushed once per
// CTA into the per-CTA partial layout that k_head_grad_reduce (head.cu) sums.
#include "cell_tc.cuh"

namespace regt {
using namespace tc;

namespace {
constexpr int HH = 64;                 // hidden width this kernel is built for
constexpr int OP = 16;                 // padded output_dim
constexpr int NEPI_WARPS = 8, NEPI = 256, WARP_MMA = 8, NTHREADS = NEPI + 32;
constexpr int FMT = FMT_BF16;
// shared-memory image (bytes)
constexpr int W1K = 0;                          // [n=128][k=64]  SW128, rows 128      B of M1
constexpr int W1TK = W1K + 128 * 128;           // [n=64][k=128]  SW128, rows 64, 2 blk B of M4
constexpr int W2K = W1TK + 2 * 64 * 128;        // [n=16][k=128]  SW128, rows 16, 2 blk B of M2
constexpr int W2TK = W2K + 2 * 16 * 128;        // [n=128][k=16]  chunk tile            B of M3
constexpr int T_A0 = W2TK + 2 * 128 * 16;       // [128][64]  relu(hid)   SW128 (1 block)
constexpr int T_A1 = T_A0 + 128 * 128;          // [128][128] a1          SW128 (2 blocks)
constexpr int T_D1 = T_A1 + 2 * 128 * 128;      // [128][128] d a1        SW128 (2 blocks)
constexpr int T_DO = T_D1 + 2 * 128 * 128;      // [128][16]  d out       chunk tile (2 chunks)
constexpr int T_ONE = T_DO + 2 * 128 * 16;      // [128][16]  col 0 = 1   chunk tile (2 chunks)
constexpr int C_B = T_ONE + 2 * 128 * 16;       // b1[128] | b2[16] fp32
constexpr int SMEM_BYTES = C_B + (128 + 16) * 4;
// TMEM columns
constexpr int C_A1 = 0, C_OUT = 128, C_G = 160, C_DW1 = 224, C_DB1 = 288, C_DW2 = 304;

struct HeadTcArgs {
  long long BN;
  int O, ntc, nqt;
  float scale;
  const float *w1, *w2, *b1, *b2;        // linear1.weight [128][64], linear2.weight [O][128]
  const float* hid_part;                 // [ntc][nqt][16][128][4] attention partials of the cell (NULL: hid_in is final)
  const float* hid_in;
  float* hid_out;                        // out_hidden [BN][64]
  const float* y;
  const float* d_hidden;
  float *out, *d_out, *G, *hpart;
  int part_stride;
  LossX lx;
};

__device__ __forceinline__ void put_bf16(uint8_t* base, uint32_t off, float v) {
  *reinterpret_cast<__nv_bfloat16*>(base + off) = __float2bfloat16(v);
}
}  // namespace

template <bool LX>
__global__ void __launch_bounds__(NTHREADS, 1) k_head_tc(HeadTcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_a0, bar_m1, bar_a1, bar_m2, bar_a2, bar_m3, bar_a3, bar_m4, bar_w;
  __shared__ uint32_t tmem_base_s;
  __shared__ float red[NEPI_WARPS][12];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int O = a.O;

  if (tid == 0) {
    mbar_init(&bar_a0, NEPI); mbar_init(&bar_a1, NEPI); mbar_init(&bar_a2, NEPI); mbar_init(&bar_a3, NEPI);
    mbar_init(&bar_m1, 1); mbar_init(&bar_m2, 1); mbar_init(&bar_m3, 1); mbar_init(&bar_m4, 1); mbar_init(&bar_w, 1);
    fence_barrier_init();
  }
  if (warp == WARP_MMA) tmem_alloc(&tmem_base_s, 512);
  // ---- weight image: fp32 parameters -> bf16 operand tiles (every CTA builds its own copy) ----
  for (int i = tid; i < 128 * HH; i += NTHREADS) {       // w1[m][k]
    const int m = i / HH, k = i % HH;
    const float v = __ldg(a.w1 + i);
    put_bf16(sm + W1K, sw128_off(m, k * 2, 128), v);      // B of M1: row n = m, K = k
    put_bf16(sm + W1TK, sw128_off(k, m * 2, 64), v);      // B of M4: row n = k, K = m
  }
  for (int i = tid; i < OP * 128; i += NTHREADS) {        // w2[o][m], zero rows for o >= O
    const int o = i / 128, m = i % 128;
    const float v = o < O ? __ldg(a.w2 + (size_t)o * 128 + m) : 0.f;
    put_bf16(sm + W2K, sw128_off(o, m * 2, 16), v);       // B of M2: row n = o, K = m
    put_bf16(sm + W2TK, chunk_off(m, (o * 2) >> 4, 128) + ((o * 2) & 15), v);   // B of M3: row n = m, K = o
  }
  for (int i = tid; i < 128; i += NTHREADS) {
    reinterpret_cast<float*>(sm + C_B)[i] = __ldg(a.b1 + i);
    *reinterpret_cast<uint4*>(sm + T_ONE + chunk_off(i, 0, 128)) = make_uint4(0x00003F80u, 0, 0, 0);   // bf16 1.0 in col 0
    *reinterpret_cast<uint4*>(sm + T_ONE + chunk_off(i, 1, 128)) = make_uint4(0, 0, 0, 0);
  }
  if (tid < OP) reinterpret_cast<float*>(sm + C_B)[128 + tid] = tid < O ? __ldg(a.b2 + tid) : 0.f;
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const float* cb = reinterpret_cast<const float*>(sm + C_B);
  const int n_my = (a.nqt - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA

  if (warp < NEPI_WARPS) {
    const int r = (warp & 3) * 32 + lane;    // row of the tile = TMEM lane
    const int ch = warp >> 2;                // column half
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    float lsum = 0.f, lsc = 0.f, db2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) db2[j] = 0.f;
    for (int i = 0; i < n_my; ++i) {
      const uint32_t ph = i & 1;
      const int qt = blockIdx.x + i * gridDim.x;
      const long long q = (long long)qt * TC_ROWS + r;
      const bool valid = q < a.BN;
      // ---- P0: hid (32 columns of this thread's row) ----
      uint32_t hmask = 0;
      {
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
        if (valid) {
          if (a.hid_part) {
            for (int c = 0; c < a.ntc; ++c) {   // fixed order: deterministic; tiled partials [chunk][qt][HH/4][128][4]
              const float4* p = reinterpret_cast<const float4*>(a.hid_part) +
                                (((size_t)c * a.nqt + qt) * (HH / 4) + ch * 8) * TC_ROWS + r;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 t = __ldg(p + (size_t)j * TC_ROWS);
                v[4 * j] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w;
              }
            }
            float4* o = reinterpret_cast<float4*>(a.hid_out + q * HH + ch * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
            const float4* p = reinterpret_cast<const float4*>(a.hid_in + q * HH + ch * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 t = __ldg(p + j);
              v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          hmask |= (v[j] > 0.f ? 1u : 0u) << j;
          v[j] = fmaxf(v[j], 0.f);
        }
        if (i > 0) mbar_wait(&bar_w, (uint32_t)((i - 1) & 1));   // the previous tile's MMAs released the tiles
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 p;
          p.x = pack_bf16(v[j], v[j + 1]); p.y = pack_bf16(v[j + 2], v[j + 3]);
          p.z = pack_bf16(v[j + 4], v[j + 5]); p.w = pack_bf16(v[j + 6], v[j + 7]);
          *reinterpret_cast<uint4*>(sm + T_A0 + sw128_off(r, (ch * 32 + j) * 2, TC_ROWS)) = p;
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_a0);

      // ---- P1: a1 = relu(a1_pre + b1), 64 columns ----
      uint32_t amask[2];
      mbar_wait(&bar_m1, ph);
      tc_fence_after();
#pragma unroll
      for (int hlf = 0; hlf < 2; ++hlf) {
        const int c0 = ch * 64 + hlf * 32;
        float v[32];
        tmem_ld32(tlane + C_A1 + c0, v);
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          v[j] = fmaxf(v[j] + cb[c0 + j], 0.f);
          m |= (v[j] > 0.f ? 1u : 0u) << j;
        }
        amask[hlf] = m;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 p;
          p.x = pack_bf16(v[j], v[j + 1]); p.y = pack_bf16(v[j + 2], v[j + 3]);
          p.z = pack_bf16(v[j + 4], v[j + 5]); p.w = pack_bf16(v[j + 6], v[j + 7]);
          *reinterpret_cast<uint4*>(sm + T_A1 + sw128_off(r, (c0 + j) * 2, TC_ROWS)) = p;
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_a1);

      // ---- P2: out, loss, d_out (8 of the 16 padded outputs per thread) ----
      mbar_wait(&bar_m2, ph);
      tc_fence_after();
      {
        float v[8], dv[8];
        tmem_ld8(tlane + C_OUT + ch * 8, v);
        float inv = a.scale;
        if constexpr (LX) inv = valid ? lossx_inv(a.lx, q, a.scale) : a.scale;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int n = ch * 8 + j;
          dv[j] = 0.f;
          if (valid && n < O) {
            const float o = v[j] + cb[128 + n];
            a.out[q * O + n] = o;
            if constexpr (LX) {
              dv[j] = lossx_elem(a.lx, o, __ldg(a.y + q * O + n), inv, a.scale, lsum, lsc);
            } else {
              const float diff = o - __ldg(a.y + q * O + n);
              lsum = fmaf(diff, diff, lsum);
              dv[j] = 2.0f * diff * a.scale;
            }
            a.d_out[q * O + n] = dv[j];
            db2[j] += dv[j];
          }
        }
        uint4 p;
        p.x = pack_bf16(dv[0], dv[1]); p.y = pack_bf16(dv[2], dv[3]);
        p.z = pack_bf16(dv[4], dv[5]); p.w = pack_bf16(dv[6], dv[7]);
        *reinterpret_cast<uint4*>(sm + T_DO + chunk_off(r, ch, TC_ROWS)) = p;
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_a2);

      // ---- P3: d a1 = da1_pre * (a1 > 0), 64 columns ----
      mbar_wait(&bar_m3, ph);
      tc_fence_after();
#pragma unroll
      for (int hlf = 0; hlf < 2; ++hlf) {
        const int c0 = ch * 64 + hlf * 32;
        float v[32];
        tmem_ld32(tlane + C_A1 + c0, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = ((amask[hlf] >> j) & 1u) ? v[j] : 0.f;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 p;
          p.x = pack_bf16(v[j], v[j + 1]); p.y = pack_bf16(v[j + 2], v[j + 3]);
          p.z = pack_bf16(v[j + 4], v[j + 5]); p.w = pack_bf16(v[j + 6], v[j + 7]);
          *reinterpret_cast<uint4*>(sm + T_D1 + sw128_off(r, (c0 + j) * 2, TC_ROWS)) = p;
        }
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(&bar_a3);

      // ---- P4: G = G_pre * (hid > 0) (+ d_hidden), 32 columns, tiled layout [qt][HH/4][128][4] ----
      mbar_wait(&bar_m4, ph);
      tc_fence_after();
      {
        float v[32];
        tmem_ld32(tlane + C_G + ch * 32, v);
        if (valid) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = ((hmask >> j) & 1u) ? v[j] : 0.f;
          if (a.d_hidden) {
            const float4* p = reinterpret_cast<const float4*>(a.d_hidden + q * HH + ch * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 t = __ldg(p + j);
              v[4 * j] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w;
            }
          }
          float4* g = reinterpret_cast<float4*>(a.G) + (size_t)qt * (HH / 4) * TC_ROWS;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            g[(size_t)(ch * 8 + j) * TC_ROWS + r] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
      }
      tc_fence_before();
    }
    // ---- flush: per-CTA partials  dW1 [128][64] | dW2 [O][128] | db1 [128] | db2 [O] | loss ----
    float* hp = a.hpart + (size_t)blockIdx.x * a.part_stride;
    const int n1 = 128 * HH, n2 = O * 128;
    if (n_my > 0) {
      mbar_wait(&bar_w, (uint32_t)((n_my - 1) & 1));
      tc_fence_after();
      float v[32];
      tmem_ld32(tlane + C_DW1 + ch * 32, v);      // lane = m (row of linear1.weight), columns = k
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(hp + (size_t)r * HH + ch * 32 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      float u[8];
      tmem_ld8(tlane + C_DW2 + ch * 8, u);        // lane = m, columns = o
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (ch * 8 + j < O) hp[n1 + (size_t)(ch * 8 + j) * 128 + r] = u[j];
      if (ch == 0) {
        tmem_ld8(tlane + C_DB1, u);               // column 0 = sum over rows of d a1
        hp[n1 + n2 + r] = u[0];
      }
      tc_fence_before();
    } else {
      for (int j = 0; j < 32; ++j) hp[(size_t)r * HH + ch * 32 + j] = 0.f;
      for (int j = 0; j < 8; ++j)
        if (ch * 8 + j < O) hp[n1 + (size_t)(ch * 8 + j) * 128 + r] = 0.f;
      if (ch == 0) hp[n1 + n2 + r] = 0.f;
    }
    // db2 and the loss: warp shuffle tree, then a fixed-order sum over the warps
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      lsum += __shfl_down_sync(0xffffffffu, lsum, d);
      if constexpr (LX) lsc += __shfl_down_sync(0xffffffffu, lsc, d);
#pragma unroll
      for (int j = 0; j < 8; ++j) db2[j] += __shfl_down_sync(0xffffffffu, db2[j], d);
    }
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) red[warp][j] = db2[j];
      red[warp][8] = lsum;
      if constexpr (LX) red[warp][9] = lsc;
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory");
    if (tid < OP) {
      const int c = tid >> 3, j = tid & 7;   // outputs of column half c live in warps 4c .. 4c+3
      const float s = ((red[4 * c][j] + red[4 * c + 1][j]) + red[4 * c + 2][j]) + red[4 * c + 3][j];
      if (tid < O) hp[n1 + n2 + 128 + tid] = s;
    } else if (tid == 32) {
      float s = 0.f;
#pragma unroll
      for (int w8 = 0; w8 < NEPI_WARPS; ++w8) s += red[w8][8];
      if constexpr (LX) {
        float s2 = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < NEPI_WARPS; ++w8) s2 += red[w8][9];
        hp[n1 + n2 + 128 + O] = s * a.scale + s2;
      } else {
        hp[n1 + n2 + 128 + O] = s * a.scale;
      }
    }
  } else {
    // ================= MMA issuer =================
    const uint32_t base = smem_u32(sm);
    const uint32_t id_a1 = make_idesc(FMT, 128, 128, 0, 0), id_out = make_idesc(FMT, 128, OP, 0, 0),
                   id_g = make_idesc(FMT, 128, HH, 0, 0);
    const uint32_t id_w1 = make_idesc(FMT, 128, HH, 1, 1), id_w16 = make_idesc(FMT, 128, OP, 1, 1);
    constexpr int BLK = TC_ROWS * 128;   // one 128-byte-wide swizzle block of a 128-row tile
    for (int i = 0; i < n_my; ++i) {
      const uint32_t ph = i & 1, accw = i > 0 ? 1u : 0u;
      mbar_wait(&bar_a0, ph);
      tc_fence_after();
      if (lane == 0) {   // M1: a1_pre = A0 . W1^T   (K = 64)
#pragma unroll
        for (int k = 0; k < HH / 16; ++k)
          umma<FMT>(tmem + C_A1, make_desc(base + T_A0 + k * 32, 16, 1024, LAYOUT_SW128),
                    make_desc(base + W1K + k * 32, 16, 1024, LAYOUT_SW128), id_a1, k > 0 ? 1u : 0u);
        umma_commit(&bar_m1);
      }
      __syncwarp();
      mbar_wait(&bar_a1, ph);
      tc_fence_after();
      if (lane == 0) {   // M2: out = A1 . W2^T   (K = 128: two swizzle blocks)
#pragma unroll
        for (int k = 0; k < 128 / 16; ++k) {
          const int kb = k * 32;
          umma<FMT>(tmem + C_OUT, make_desc(base + T_A1 + (kb >> 7) * BLK + (kb & 127), 16, 1024, LAYOUT_SW128),
                    make_desc(base + W2K + (kb >> 7) * 16 * 128 + (kb & 127), 16, 1024, LAYOUT_SW128), id_out,
                    k > 0 ? 1u : 0u);
        }
        umma_commit(&bar_m2);
      }
      __syncwarp();
      mbar_wait(&bar_a2, ph);
      tc_fence_after();
      if (lane == 0) {   // M3: da1_pre = Do . W2   (K = 16, one step of two 16-byte chunks)
        umma<FMT>(tmem + C_A1, make_desc(base + T_DO, TC_ROWS * 16, 128, LAYOUT_NONE),
                  make_desc(base + W2TK, 128 * 16, 128, LAYOUT_NONE), id_a1, 0u);
        umma_commit(&bar_m3);
        // dW2^T[m][o] += sum_rows A1[row][m] Do[row][o]   (MN-major operands, K = the 128 rows)
#pragma unroll
        for (int k = 0; k < TC_ROWS / 16; ++k)
          umma<FMT>(tmem + C_DW2, make_desc(base + T_A1 + k * 2048, BLK, 1024, LAYOUT_SW128),
                    make_desc(base + T_DO + k * 256, 128, TC_ROWS * 16, LAYOUT_NONE), id_w16, (k > 0) ? 1u : accw);
      }
      __syncwarp();
      mbar_wait(&bar_a3, ph);
      tc_fence_after();
      if (lane == 0) {   // M4: G_pre = D1 . W1   (K = 128)
#pragma unroll
        for (int k = 0; k < 128 / 16; ++k) {
          const int kb = k * 32;
          umma<FMT>(tmem + C_G, make_desc(base + T_D1 + (kb >> 7) * BLK + (kb & 127), 16, 1024, LAYOUT_SW128),
                    make_desc(base + W1TK + (kb >> 7) * 64 * 128 + (kb & 127), 16, 1024, LAYOUT_SW128), id_g,
                    k > 0 ? 1u : 0u);
        }
        umma_commit(&bar_m4);
        // dW1[m][k] += sum_rows D1[row][m] A0[row][k] ;  db1[m] += sum_rows D1[row][m] * 1
#pragma unroll
        for (int k = 0; k < TC_ROWS / 16; ++k) {
          const uint64_t da = make_desc(base + T_D1 + k * 2048, BLK, 1024, LAYOUT_SW128);
          umma<FMT>(tmem + C_DW1, da, make_desc(base + T_A0 + k * 2048, BLK, 1024, LAYOUT_SW128), id_w1, (k > 0) ? 1u : accw);
          umma<FMT>(tmem + C_DB1, da, make_desc(base + T_ONE + k * 256, 128, TC_ROWS * 16, LAYOUT_NONE), id_w16,
                    (k > 0) ? 1u : accw);
        }
        umma_commit(&bar_w);
      }
      __syncwarp();
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == WARP_MMA) tmem_dealloc(tmem, 512);
}

bool head_tc_fits(int H, int O) { return H == HH && O <= OP; }
int head_tc_grid(const regt_args* a) {
  const long long BN = (long long)a->B * a->N;
  return (int)min((long long)148, (BN + TC_ROWS - 1) / TC_ROWS);
}
// the bf16 cell left per-chunk partials of out_hidden (Route::hid_partials): summed here while loading the tiles
int head_forward_tc(const regt_args* a, const Layout& L, cudaStream_t st) {
  HeadTcArgs k{};
  k.BN = (long long)a->B * a->N;
  k.O = a->O;
  k.nqt = (int)((k.BN + TC_ROWS - 1) / TC_ROWS);
  k.scale = 1.0f / ((float)(a->loss_nodes > 0 ? a->loss_nodes : a->N) * (float)a->O);
  k.w1 = a->p.head_w1; k.w2 = a->p.head_w2; k.b1 = a->p.head_b1; k.b2 = a->p.head_b2;
  k.hid_part = L.hid_part;
  k.ntc = tc_num_chunks(a);
  k.hid_in = a->out_hidden; k.hid_out = a->out_hidden;
  k.y = a->y; k.d_hidden = a->d_hidden;
  k.out = a->out; k.d_out = a->d_out; k.G = L.G; k.hpart = L.hpart;
  k.part_stride = head_part_stride_host(a->H, a->O);
  k.lx = make_lossx(a, L);
  const size_t smem = SMEM_BYTES + 1024;
  auto kern = loss_ext(a) ? k_head_tc<true> : k_head_tc<false>;
  REGT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<head_tc_grid(a), NTHREADS, smem, st>>>(k);
  REGT_LAUNCHED("k_head_tc", st);
  return 0;
}

}  // namespace regt
