// TMA-fed 3xTF32 GEMMs.
//
// A single producer thread keeps whole pipeline stages in flight with cp.async.bulk.tensor (TMA, SWIZZLE_128B boxes
// landing directly in the UMMA operand layout), converter warps do the tf32 hi/lo split in shared memory, one thread issues
// the tcgen05 MMAs into TMEM, and epilogue warps drain the accumulators.  (Loader warps that pulled the operands through
// registers, one chunk ahead, kept ~36 KB in flight per SM and ran latency-bound at 20-35 % of the HBM / tensor roofline.)
//
//   gemm_nt : C[M][N] = A[M][K] . Bt[N][K]^T
//             A chunks [128 rows][32 k] arrive as fp32; the converters overwrite them with hi = tf32(a) and write
//             lo = a - hi next to them (same swizzled position, no address arithmetic).  Bt is a weight matrix: it is
//             split ONCE into dense hi / lo arrays (k_split_hilo) and either parked in shared memory for the whole
//             kernel (N <= 128 and K <= 128: "resident") or streamed by TMA next to the A chunks.
//   gemm_tn : Cp[z][K][N] = sum over the rows r of split z of A[r][K]^T . B[r][N]   (+ the 32-column plane B2)
//             Raw [32 rows][32 cols] boxes land swizzled (conflict-free 16-byte reads); the converters transpose
//             them into K-major hi / lo tiles.  One launch may cover several column segments of A, each with its own
//             B operand and output (all four gate-gradient blocks of D in one grid that fills the SMs).
#include <cuda.h>   // CUtensorMap and its enums only: the encoder is fetched through the runtime (no libcuda link)

#include "cell_tc.cuh"

namespace regt {
using namespace tc;

namespace {
constexpr int KC = 32;               // contraction chunk: 32 fp32 = one 128-byte swizzle row
constexpr int TILE = 128 * 128;      // [128 rows][128 B] operand tile
constexpr int MAXS = 6;              // pipeline stages (upper bound)
constexpr int SMEM_BUDGET = 227 * 1024 - 1024;   // dynamic shared memory minus the 1024-byte alignment slack

__device__ __forceinline__ uint32_t tf32_rn(float a) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(a));
  return u;
}
__device__ __forceinline__ void split4(const float4 v, float4& hi, float4& lo) {
  hi.x = __uint_as_float(tf32_rn(v.x)); hi.y = __uint_as_float(tf32_rn(v.y));
  hi.z = __uint_as_float(tf32_rn(v.z)); hi.w = __uint_as_float(tf32_rn(v.w));
  lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
}
// one box of a 2-D tensor map -> shared memory; completion is counted in bytes on `bar`
__device__ __forceinline__ void tma_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmap_prefetch(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn encoder() {
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeFn)p;
  }
  return fn;
}
// fp32 [rows][cols] window of a row-major array with pitch ld (floats); boxes of box_rows x 32 floats, 128-byte swizzle,
// out-of-range elements read as zero
int tmap_2d(CUtensorMap* m, const float* base, long long cols, long long rows, long long ld, int box_rows, const char* who) {
  EncodeFn enc = encoder();
  REGT_CHECK(enc != nullptr, "%s: cuTensorMapEncodeTiled is not available from this driver", who);
  REGT_CHECK(((uintptr_t)base % 16 == 0) && ld % 4 == 0, "%s: TMA operands need 16-byte aligned base and pitch", who);
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  REGT_CHECK(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed (%d) cols=%lld rows=%lld ld=%lld", who, (int)r, cols, rows, ld);
  return 0;
}

// ------------------------------------------------------------------------------------------
// dense hi / lo images of a weight operand: hi[n][k] = tf32(B[n][k]), lo = B - hi, zero-padded to [Np][Kp]
// ------------------------------------------------------------------------------------------
__global__ void k_split_hilo(const float* __restrict__ B, long long ldb, int N, int K, int Np, int Kp, float* __restrict__ hi,
                             float* __restrict__ lo) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)Np * Kp) return;
  const int n = (int)(i / Kp), k = (int)(i - (long long)n * Kp);
  const float v = (n < N && k < K) ? __ldg(B + (size_t)n * ldb + k) : 0.f;
  const float h = __uint_as_float(tf32_rn(v));
  hi[i] = h;
  lo[i] = v - h;
}

// ------------------------------------------------------------------------------------------
// gemm_nt
// ------------------------------------------------------------------------------------------
struct NtArgs {
  CUtensorMap ta, tbh, tbl;   // A [M][K]; Bt hi / lo [Np][Kp]
  float* C;
  long long M, ldc;
  int N, K;
  int resident;               // Bt hi/lo parked in shared memory for the whole kernel
  int ns;                     // pipeline stages
};
constexpr int NT_CONV = 256;                    // converter threads (warps 0-7)
constexpr int NT_W_TMA = NT_CONV / 32;          // producer warp
constexpr int NT_W_MMA = NT_W_TMA + 1;          // MMA issuer (owns the TMEM allocation)
constexpr int NT_W_EPI = NT_W_MMA + 1;          // 4 epilogue warps
constexpr int NT_THREADS = (NT_W_EPI + 4) * 32;

// ------------------------------------------------------------------------------------------
// gemm_nt, A operand through TMEM ("TS" MMAs).  With the weight operand parked in shared memory (128 KB at N = K = 128) a
// version that kept [A hi | A lo] in shared memory had room for 3 stages = 48 KB of TMA loads in flight and ran at 55 % of
// the HBM bandwidth (measured in round 1, since removed).  Here the converters write hi / lo straight into TMEM
// (tcgen05.st, 4 slots x 64 columns next to the two 128-column accumulators), the MMAs read A from there, and shared
// memory holds only RAW fp32 chunks: 6 stages x 16 KB in flight (H = 128: 1.11 -> 0.88 ms, 4.5 TB/s = 68 % of the
// measured HBM peak).  Streamed weights (N or K > 128): a stage is [raw A | B hi | B lo] = 48 KB, four of them.
// ------------------------------------------------------------------------------------------
constexpr int TS_SLOTS = 4;      // A (hi | lo) slots in TMEM, 64 columns each, after the two accumulators
__global__ void __launch_bounds__(NT_THREADS, 1) k_gemm_nt_tma_ts(const __grid_constant__ NtArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_tma[MAXS], bar_rfree[MAXS], bar_afull[TS_SLOTS], bar_afree[TS_SLOTS], bar_b, bar_acc_full[2], bar_acc_free[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ns = a.ns;
  const int nchunks = (a.K + KC - 1) / KC;
  const int ntn = (a.N + 127) / 128;
  const long long ntiles = ((a.M + 127) / 128) * ntn;
  const int stage_bytes = a.resident ? TILE : 3 * TILE;           // raw fp32 A chunk ( | B hi | B lo when the weights stream)
  uint8_t* bres = sm;
  uint8_t* stages = sm + (a.resident ? nchunks * 2 * TILE : 0);
  if (tid == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(&bar_tma[s], 1);
      mbar_init(&bar_rfree[s], a.resident ? NT_CONV : NT_CONV + 1);   // streamed weights: + the commit of the MMAs that read them
    }
    for (int s = 0; s < TS_SLOTS; ++s) {
      mbar_init(&bar_afull[s], NT_CONV);
      mbar_init(&bar_afree[s], 1);
    }
    mbar_init(&bar_b, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bar_acc_full[b], 1);
      mbar_init(&bar_acc_free[b], 128);
    }
    fence_barrier_init();
  }
  if (warp == NT_W_MMA) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t tmem_a = tmem + 256;              // slot s: hi at columns 64 s .. +31, lo at 64 s + 32 .. +63

  if (warp < NT_W_TMA) {
    // ---- converters: thread = (row of the tile, half of the chunk's 32 k values); the two warps of a TMEM lane quarter
    //      take one half each.  Raw rows are 128-byte swizzled: the 8 lanes of a quarter-warp read 8 different banks groups.
    const int q = warp & 3, half = warp >> 2;
    const int r = q * 32 + lane;
    const uint32_t tl = tmem_a + ((uint32_t)(q * 32) << 16) + 16 * half;
    long long gc = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      for (int kc = 0; kc < nchunks; ++kc, ++gc) {
        const int s = (int)(gc % ns), sl = (int)(gc % TS_SLOTS);
        mbar_wait(&bar_tma[s], (uint32_t)((gc / ns) & 1));
        const uint8_t* rw = stages + (size_t)s * stage_bytes + r * 128;
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float4 v = *reinterpret_cast<const float4*>(rw + (((half * 4 + c) ^ (r & 7)) << 4));
          float4 h, l;
          split4(v, h, l);
          hi[4 * c] = __float_as_uint(h.x); hi[4 * c + 1] = __float_as_uint(h.y); hi[4 * c + 2] = __float_as_uint(h.z); hi[4 * c + 3] = __float_as_uint(h.w);
          lo[4 * c] = __float_as_uint(l.x); lo[4 * c + 1] = __float_as_uint(l.y); lo[4 * c + 2] = __float_as_uint(l.z); lo[4 * c + 3] = __float_as_uint(l.w);
        }
        // the raw stage may be refilled once every converter has arrived; an arrive does not wait for this thread's loads
        // (see k_gemm_tn_tma), so it sits behind a branch on the loaded values
        if ((hi[0] | hi[4] | hi[8] | hi[12]) == 0x7FC0DEADu) __nanosleep(1);
        mbar_arrive(&bar_rfree[s]);
        if (gc >= TS_SLOTS) {
          mbar_wait(&bar_afree[sl], (uint32_t)((gc / TS_SLOTS - 1) & 1));
          tc_fence_after();
        }
        tmem_st16(tl + 64 * sl, hi);
        tmem_st16(tl + 64 * sl + 32, lo);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&bar_afull[sl]);
      }
    }
  } else if (warp == NT_W_TMA) {
    if (lane == 0) {
      tmap_prefetch(&a.ta);
      tmap_prefetch(&a.tbh);
      tmap_prefetch(&a.tbl);
      if (a.resident) {
        mbar_arrive_expect_tx(&bar_b, (uint32_t)(nchunks * 2 * TILE));
        for (int kc = 0; kc < nchunks; ++kc) {
          tma_2d(bres + (size_t)kc * 2 * TILE, &a.tbh, kc * KC, 0, &bar_b);
          tma_2d(bres + (size_t)kc * 2 * TILE + TILE, &a.tbl, kc * KC, 0, &bar_b);
        }
      }
      long long gc = 0;
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int m0 = (int)((tile / ntn) * 128), n0 = (int)(tile % ntn) * 128;
        for (int kc = 0; kc < nchunks; ++kc, ++gc) {
          const int s = (int)(gc % ns);
          if (gc >= ns) mbar_wait(&bar_rfree[s], (uint32_t)((gc / ns - 1) & 1));
          uint8_t* st = stages + (size_t)s * stage_bytes;
          mbar_arrive_expect_tx(&bar_tma[s], (uint32_t)stage_bytes);
          tma_2d(st, &a.ta, kc * KC, m0, &bar_tma[s]);
          if (!a.resident) {
            tma_2d(st + TILE, &a.tbh, kc * KC, n0, &bar_tma[s]);
            tma_2d(st + 2 * TILE, &a.tbl, kc * KC, n0, &bar_tma[s]);
          }
        }
      }
    }
  } else if (warp == NT_W_MMA) {
    const uint32_t bres0 = smem_u32(bres), stage0 = smem_u32(stages);
    if (a.resident) mbar_wait(&bar_b, 0);
    long long gc = 0, li = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++li) {
      const int nt = min(128, a.N - (int)(tile % ntn) * 128);
      const uint32_t idesc = make_idesc(FMT_TF32, 128, nt, 0, 0);
      const int buf = (int)(li & 1);
      if (li >= 2) {
        mbar_wait(&bar_acc_free[buf], (uint32_t)((li / 2 - 1) & 1));
        tc_fence_after();
      }
      for (int kc = 0; kc < nchunks; ++kc, ++gc) {
        const int sl = (int)(gc % TS_SLOTS);
        mbar_wait(&bar_afull[sl], (uint32_t)((gc / TS_SLOTS) & 1));
        tc_fence_after();
        if (lane == 0) {
          const uint32_t ah = tmem_a + 64 * sl, al = ah + 32;
          const int s = (int)(gc % ns);
          const uint32_t bt = a.resident ? bres0 + kc * 2 * TILE : stage0 + s * stage_bytes + TILE;
#pragma unroll
          for (int p = 0; p < 3; ++p) {   // hi*hi, lo*hi, hi*lo
            const uint32_t ap = (p == 1) ? al : ah, bp = bt + (p == 2 ? TILE : 0);
#pragma unroll
            for (int k = 0; k < KC / 8; ++k)
              umma_ts_tf32(tmem + buf * 128, ap + 8 * k, make_desc(bp + k * 32, 16, 1024, LAYOUT_SW128), idesc,
                           (kc > 0 || p > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&bar_afree[sl]);
          if (!a.resident) umma_commit(&bar_rfree[s]);   // the streamed weight tiles of this stage have been read
          if (kc + 1 == nchunks) umma_commit(&bar_acc_full[buf]);
        }
        __syncwarp();
      }
    }
    tc_fence_before();
  } else {
    // ---- epilogue warps: TMEM -> registers -> C (thread = row of the tile) ----
    const int r = (warp & 3) * 32 + lane;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    long long li = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++li) {
      const int buf = (int)(li & 1);
      const int n0 = (int)(tile % ntn) * 128;
      const int nt = min(128, a.N - n0);
      const long long arow = (tile / ntn) * 128 + r;
      const bool a_ok = arow < a.M;
      float* cp = a.C + (a_ok ? arow : 0) * a.ldc + n0;
      mbar_wait(&bar_acc_full[buf], (uint32_t)((li / 2) & 1));
      tc_fence_after();
      for (int c0 = 0; c0 < nt; c0 += 32) {
        float v[32];
        if (c0 + 32 <= nt) {
          tmem_ld32(tlane + buf * 128 + c0, v);
        } else {
          float u[16];
          tmem_ld16(tlane + buf * 128 + c0, u);
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = u[j];
        }
        if (a_ok) {
          const int w = min(32, nt - c0);
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            if (j < w) *reinterpret_cast<float4*>(cp + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(&bar_acc_free[buf]);
    }
  }
  __syncthreads();
  if (warp == NT_W_MMA) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// gemm_tn
// ------------------------------------------------------------------------------------------
struct TnSeg {
  int k0, k1;   // columns [k0, k1) of A
  int b;        // B operand of this segment: index into tb[], or -1 (only the B2 plane)
  float* C;     // [split][k1 - k0][N]
};
struct TnArgs {
  CUtensorMap ta, tb[2], tf;   // A [M][Ktot], B operands [M][N], B2 [M][32]
  TnSeg seg[4];
  int nseg;
  float* C2;                   // [split][Ktot][32] (stride c2_split between splits)
  long long c2_split;
  long long M, chunk;          // rows contracted over; rows per split (multiple of 32)
  int N, N2;
  int relu_b;                  // the B operands are read through max(., 0)
};
constexpr int TN_CONV = 256;                  // converter / epilogue threads (warps 0-7)
constexpr int TN_W_MMA = TN_CONV / 32;
constexpr int TN_W_TMA = TN_W_MMA + 1;
constexpr int TN_THREADS = (TN_W_TMA + 1) * 32;
constexpr int TN_NR = 2, TN_NC = 2;           // raw (TMA) stages, converted (MMA operand) stages
constexpr int TN_BOX = 32 * 128;              // one [32 rows][32 cols] fp32 box
constexpr int TN_RAW = 9 * TN_BOX;            // A: 4 boxes, B: 4 boxes, B2: 1 box
constexpr int TN_BT = (128 + 32) * 128;       // converted B tile with the 32 extra feature rows
constexpr int TN_CV = 2 * TILE + 2 * TN_BT;   // A hi | A lo | B hi | B lo
// The tensor core's fp32 accumulation is not round-to-nearest: its error grows linearly with the number of MMAs
// chained into one accumulator (measured ~2e-8 relative per MMA).  A row contraction chains 12 MMAs per chunk over up to
// 10^5 rows, so the TMEM accumulator is drained into fp32 registers (round-to-nearest adds) every TN_GROUP chunks; two
// accumulators alternate so the drain of group g runs under the MMAs of group g + 1.
constexpr int TN_GROUP = 8;
constexpr int TN_ACC = 256;                   // TMEM column stride between the two accumulators (each 128 + 32 feature columns wide)
static_assert(TN_NR * TN_RAW + TN_NC * TN_CV <= SMEM_BUDGET, "gemm_tn stages exceed shared memory");

__global__ void __launch_bounds__(TN_THREADS, 1) k_gemm_tn_tma(const __grid_constant__ TnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_raw[TN_NR], bar_rfree[TN_NR], bar_full[TN_NC], bar_empty[TN_NC], bar_done, bar_acc_free[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kg = blockIdx.x * 128;   // first column of A of this tile
  int si = 0;
  for (int s = 1; s < a.nseg; ++s)
    if (kg >= a.seg[s].k0) si = s;
  const int sk0 = a.seg[si].k0, sk1 = a.seg[si].k1, sb = a.seg[si].b;
  float* segC = a.seg[si].C;
  const int n0 = blockIdx.y * 128;
  const int kt = min(128, sk1 - kg);                                    // output rows of this tile (multiple of 32)
  const int nt = sb >= 0 ? max(0, min(128, a.N - n0)) : 0;              // columns from the B operand
  const int n2 = (blockIdx.y == 0) ? a.N2 : 0;                          // + the 32 feature columns on N tile 0
  const int ntot = nt + n2;
  const long long r0 = (long long)blockIdx.z * a.chunk, r1 = min(a.M, r0 + a.chunk);
  const int nchunks = ntot > 0 ? (int)max(0ll, (r1 - r0 + KC - 1) / KC) : 0;
  uint8_t* raw = sm;
  uint8_t* cv = sm + TN_NR * TN_RAW;
  if (tid == 0) {
    for (int s = 0; s < TN_NR; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_rfree[s], TN_CONV);
    }
    for (int s = 0; s < TN_NC; ++s) {
      mbar_init(&bar_full[s], TN_CONV);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_done, 1);
    mbar_init(&bar_acc_free[0], TN_CONV);
    mbar_init(&bar_acc_free[1], TN_CONV);
    fence_barrier_init();
  }
  if (warp == TN_W_MMA) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const int ablk = kt / 32, bblk = (nt + 31) / 32;   // boxes per chunk

  if (warp < TN_W_MMA) {
    // ---- converters: warp (w & 3) owns column block w & 3 of A and of B, its half w >> 2 four float4s of that block;
    //      lane = row of the chunk.  The raw boxes are 128-byte swizzled, so the eight lanes of a quarter-warp read
    //      eight different 16-byte columns; the transposed 4-byte stores of one (c, e) hit 32 different banks. ----
    const int blk = warp & 3, half = warp >> 2;
    const bool a_ok = blk < ablk, b_ok = blk < bblk;
    // running sums of this thread's part of the output tile: row orow, 16-column groups half, half + 2, ...
    const int orow = (warp & 3) * 32 + lane;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    float acc[5][16];
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[i][j] = 0.f;
    int drained = 0;
    auto drain = [&](int buf) {
      tc_fence_after();
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int c0 = half * 16 + 32 * i;
        if (c0 < ntot) {
          float v[16];
          tmem_ld16(tlane + buf * TN_ACC + c0, v);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[i][j] += v[j];
        }
      }
      tc_fence_before();
      mbar_arrive(&bar_acc_free[buf]);
    };
    for (int kc = 0; kc < nchunks; ++kc) {
      const int rs = kc % TN_NR, cs = kc % TN_NC;
      mbar_wait(&bar_raw[rs], (uint32_t)((kc / TN_NR) & 1));
      const uint8_t* rw = raw + rs * TN_RAW;
      float4 av[4], bv[4], fv = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint32_t off = (uint32_t)(lane * 128 + (((half * 4 + c) ^ (lane & 7)) << 4));
        av[c] = a_ok ? *reinterpret_cast<const float4*>(rw + blk * TN_BOX + off) : make_float4(0.f, 0.f, 0.f, 0.f);
        bv[c] = b_ok ? *reinterpret_cast<const float4*>(rw + (4 + blk) * TN_BOX + off) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (a.relu_b) {
#pragma unroll
        for (int c = 0; c < 4; ++c) bv[c] = make_float4(fmaxf(bv[c].x, 0.f), fmaxf(bv[c].y, 0.f), fmaxf(bv[c].z, 0.f), fmaxf(bv[c].w, 0.f));
      }
      if (n2) fv = *reinterpret_cast<const float4*>(rw + 8 * TN_BOX + lane * 128 + ((warp ^ (lane & 7)) << 4));
      {   // The raw stage is refilled by TMA once all 256 threads have arrived, and an mbarrier arrive does NOT wait for
          // this thread's earlier shared-memory loads to return (observed on B200: the tail loads of a warp read the
          // NEXT chunk's bytes).  A branch on the loaded values forces their completion before the arrive issues.
        const uint32_t dep = __float_as_uint(av[0].x) | __float_as_uint(av[1].x) | __float_as_uint(av[2].x) | __float_as_uint(av[3].x) |
                             __float_as_uint(bv[0].x) | __float_as_uint(bv[1].x) | __float_as_uint(bv[2].x) | __float_as_uint(bv[3].x) |
                             __float_as_uint(fv.x);
        if (dep == 0x7FC0DEADu) __nanosleep(1);
        mbar_arrive(&bar_rfree[rs]);
      }
      if (kc >= TN_NC) mbar_wait(&bar_empty[cs], (uint32_t)((kc / TN_NC - 1) & 1));
      // the MMAs of chunks <= kc - TN_NC have completed: group g is whole once (g + 1) * TN_GROUP - 1 <= kc - TN_NC
      if (kc >= TN_GROUP + TN_NC - 1 && (kc - (TN_NC - 1)) % TN_GROUP == 0) {
        drain(drained & 1);
        ++drained;
      }
      uint8_t* st = cv + cs * TN_CV;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 hi, lo;
        split4(av[c], hi, lo);
        const float ah[4] = {hi.x, hi.y, hi.z, hi.w}, al[4] = {lo.x, lo.y, lo.z, lo.w};
        split4(bv[c], hi, lo);
        const float bh[4] = {hi.x, hi.y, hi.z, hi.w}, bl[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = blk * 32 + 16 * half + 4 * c + e;
          const uint32_t off = sw128_off(col, lane * 4, 128);
          *reinterpret_cast<float*>(st + off) = ah[e];
          *reinterpret_cast<float*>(st + TILE + off) = al[e];
          if (col < nt) {   // rows nt.. of the B tile belong to the feature columns
            *reinterpret_cast<float*>(st + 2 * TILE + off) = bh[e];
            *reinterpret_cast<float*>(st + 2 * TILE + TN_BT + off) = bl[e];
          }
        }
      }
      if (n2) {   // feature columns: B tile rows nt + 4*warp + e
        float4 hi, lo;
        split4(fv, hi, lo);
        const float fh[4] = {hi.x, hi.y, hi.z, hi.w}, fl[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const uint32_t off = sw128_off(nt + 4 * warp + e, lane * 4, 128);
          *reinterpret_cast<float*>(st + 2 * TILE + off) = fh[e];
          *reinterpret_cast<float*>(st + 2 * TILE + TN_BT + off) = fl[e];
        }
      }
      fence_proxy_async();
      mbar_arrive(&bar_full[cs]);
    }
    // ---- epilogue: remaining groups, then the partial tile -> Cp[z] (an empty split contributes zeros) ----
    const int ngroups = (nchunks + TN_GROUP - 1) / TN_GROUP;
    if (nchunks > 0) mbar_wait(&bar_done, 0);
    for (; drained < ngroups; ++drained) drain(drained & 1);
    const bool row_ok = orow < kt;
    float* cp = nt > 0 ? segC + ((size_t)blockIdx.z * (sk1 - sk0) + (kg - sk0) + (row_ok ? orow : 0)) * a.N + n0 : nullptr;
    float* cp2 = n2 ? a.C2 + (size_t)blockIdx.z * a.c2_split + (size_t)(kg + (row_ok ? orow : 0)) * 32 : nullptr;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int c0 = half * 16 + 32 * i;
      if (c0 < ntot && row_ok) {
        float* o = c0 < nt ? cp + c0 : cp2 + (c0 - nt);
#pragma unroll
        for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[i][j], acc[i][j + 1], acc[i][j + 2], acc[i][j + 3]);
      }
    }
  } else if (warp == TN_W_MMA) {
    const uint32_t idesc = make_idesc(FMT_TF32, 128, max(ntot, 16), 0, 0);
    const uint32_t base = smem_u32(cv);
    for (int kc = 0; kc < nchunks; ++kc) {
      const int s = kc % TN_NC;
      const int g = kc / TN_GROUP, buf = g & 1, kg0 = kc % TN_GROUP;
      if (kg0 == 0 && g >= 2) {   // the converters have drained this accumulator's previous group (g - 2)
        mbar_wait(&bar_acc_free[buf], (uint32_t)((g / 2 - 1) & 1));
        tc_fence_after();
      }
      mbar_wait(&bar_full[s], (uint32_t)((kc / TN_NC) & 1));
      tc_fence_after();
      if (lane == 0) {
        const uint32_t st = base + s * TN_CV;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const uint32_t at = st + (p == 1 ? TILE : 0), bt = st + 2 * TILE + (p == 2 ? TN_BT : 0);
#pragma unroll
          for (int k = 0; k < KC / 8; ++k)
            umma<FMT_TF32>(tmem + buf * TN_ACC, make_desc(at + k * 32, 16, 1024, LAYOUT_SW128), make_desc(bt + k * 32, 16, 1024, LAYOUT_SW128),
                           idesc, (kg0 > 0 || p > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&bar_empty[s]);
        if (kc + 1 == nchunks) umma_commit(&bar_done);
      }
      __syncwarp();
    }
    tc_fence_before();
  } else {
    // ---- producer ----
    if (lane == 0 && nchunks > 0) {
      tmap_prefetch(&a.ta);
      if (sb >= 0) tmap_prefetch(&a.tb[sb]);
      if (n2) tmap_prefetch(&a.tf);
      const uint32_t bytes = (uint32_t)((ablk + bblk + (n2 ? 1 : 0)) * TN_BOX);
      for (int kc = 0; kc < nchunks; ++kc) {
        const int rs = kc % TN_NR;
        if (kc >= TN_NR) mbar_wait(&bar_rfree[rs], (uint32_t)((kc / TN_NR - 1) & 1));
        uint8_t* rw = raw + rs * TN_RAW;
        const int row = (int)(r0 + (long long)kc * KC);
        mbar_arrive_expect_tx(&bar_raw[rs], bytes);
        for (int b = 0; b < ablk; ++b) tma_2d(rw + b * TN_BOX, &a.ta, kg + b * 32, row, &bar_raw[rs]);
        for (int b = 0; b < bblk; ++b) tma_2d(rw + (4 + b) * TN_BOX, &a.tb[sb], n0 + b * 32, row, &bar_raw[rs]);
        if (n2) tma_2d(rw + 8 * TN_BOX, &a.tf, 0, row, &bar_raw[rs]);
      }
    }
  }
  __syncthreads();
  if (warp == TN_W_MMA) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// gemm_kt: the same row contraction over TRANSPOSED tiles.  The fused cell backward (cell_f.cu) stores its gate gradients and
// the h / h*R planes as [tile][column][128 rows] -- the layout its row-per-lane epilogue threads write as whole 128-byte
// lines -- and a [column][row] tile is already the K-major operand of this contraction (K = rows).  A chunk (32 rows of one
// tile) is three plain TMA boxes, [128 cols][32 k] of A^T, [N cols][32 k] of B^T and [32][32 k] of the feature plane; the
// converters only split fp32 -> tf32 hi / lo at the SAME swizzled offset (one 128-bit load and two 128-bit stores per 16
// bytes -- gemm_tn's transposing converters issue eight 4-byte stores for them and keep the LSU pipe 61 % busy).  MMA issue,
// accumulator draining and the output format are gemm_tn's.
//   A^T : [ntile][4 row quarters][Ktot][32 rows]   Ktot = 4H columns per tile    (segments of 128 columns as in gemm_tn)
//   B^T : [ntile][4][N][32]                        N <= 128 columns per tile (h or h*R)
//   F^T : [ntile][4][32][32]
// (a chunk = one row quarter of a tile: the 32 rows a warp of the producing kernel owns)
// ------------------------------------------------------------------------------------------
struct KtArgs {
  CUtensorMap ta, tb[2], tf;
  TnSeg seg[4];
  int nseg;
  float* C2;
  long long c2_split;
  long long ntile, tiles_per_split;
  int Ktot, N, N2;
};
constexpr int KT_RAW = 2 * TILE + TN_BOX;        // raw stage: A^T box | B^T box | F^T box (fp32 as loaded)

__global__ void __launch_bounds__(TN_THREADS, 1) k_gemm_kt(const __grid_constant__ KtArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_raw[TN_NR], bar_rfree[TN_NR], bar_full[TN_NC], bar_empty[TN_NC], bar_done, bar_acc_free[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kg = blockIdx.x * 128;   // first column of A^T of this M tile
  int si = 0;
  for (int s = 1; s < a.nseg; ++s)
    if (kg >= a.seg[s].k0) si = s;
  const int sk0 = a.seg[si].k0, sk1 = a.seg[si].k1, sb = a.seg[si].b;
  float* segC = a.seg[si].C;
  const int kt = min(128, sk1 - kg);                          // output rows of this tile that belong to the segment's C
  const int kt2 = min(128, a.Ktot - kg);                      // ... and to the feature outputs C2
  const int nt = sb >= 0 ? a.N : 0;                           // columns from the B operand
  const int n2 = a.N2;
  const int ntot = nt + n2;
  const long long t0 = (long long)blockIdx.z * a.tiles_per_split, t1 = min(a.ntile, t0 + a.tiles_per_split);
  const int nchunks = ntot > 0 ? (int)max(0ll, (t1 - t0) * 4) : 0;
  uint8_t* raw = sm;
  uint8_t* cv = sm + TN_NR * KT_RAW;
  if (tid == 0) {
    for (int s = 0; s < TN_NR; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_rfree[s], TN_CONV);
    }
    for (int s = 0; s < TN_NC; ++s) {
      mbar_init(&bar_full[s], TN_CONV);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_done, 1);
    mbar_init(&bar_acc_free[0], TN_CONV);
    mbar_init(&bar_acc_free[1], TN_CONV);
    fence_barrier_init();
  }
  if (warp == TN_W_MMA) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  if (warp < TN_W_MMA) {
    // ---- converters: thread = (row of the A^T / B^T tile, four of its eight 16-byte pieces); feature tile: (row tid / 8, piece tid % 8)
    const int row = (warp & 3) * 32 + lane, half = warp >> 2;
    const int frow = tid >> 3, fpc = tid & 7;
    const bool b_ok = row < nt;
    const int orow = row;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    float acc[5][16];
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[i][j] = 0.f;
    int drained = 0;
    auto drain = [&](int buf) {
      tc_fence_after();
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int c0 = half * 16 + 32 * i;
        if (c0 < ntot) {
          float v[16];
          tmem_ld16(tlane + buf * TN_ACC + c0, v);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[i][j] += v[j];
        }
      }
      tc_fence_before();
      mbar_arrive(&bar_acc_free[buf]);
    };
    uint32_t offs[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) offs[c] = (uint32_t)(row * 128 + (((half * 4 + c) ^ (row & 7)) << 4));
    const uint32_t foff = (uint32_t)(frow * 128 + ((fpc ^ (frow & 7)) << 4));
    for (int kc = 0; kc < nchunks; ++kc) {
      const int rs = kc % TN_NR, cs = kc % TN_NC;
      mbar_wait(&bar_raw[rs], (uint32_t)((kc / TN_NR) & 1));
      const uint8_t* rw = raw + rs * KT_RAW;
      float4 av[4], bv[4], fv = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        av[c] = *reinterpret_cast<const float4*>(rw + offs[c]);
        bv[c] = b_ok ? *reinterpret_cast<const float4*>(rw + TILE + offs[c]) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (n2) fv = *reinterpret_cast<const float4*>(rw + 2 * TILE + foff);
      {   // an mbarrier arrive does not wait for this thread's earlier shared-memory loads (see k_gemm_tn_tma)
        const uint32_t dep = __float_as_uint(av[0].x) | __float_as_uint(av[1].x) | __float_as_uint(av[2].x) | __float_as_uint(av[3].x) |
                             __float_as_uint(bv[0].x) | __float_as_uint(bv[1].x) | __float_as_uint(bv[2].x) | __float_as_uint(bv[3].x) |
                             __float_as_uint(fv.x);
        if (dep == 0x7FC0DEADu) __nanosleep(1);
        mbar_arrive(&bar_rfree[rs]);
      }
      if (kc >= TN_NC) mbar_wait(&bar_empty[cs], (uint32_t)((kc / TN_NC - 1) & 1));
      if (kc >= TN_GROUP + TN_NC - 1 && (kc - (TN_NC - 1)) % TN_GROUP == 0) {
        drain(drained & 1);
        ++drained;
      }
      uint8_t* st = cv + cs * TN_CV;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float4 hi, lo;
        split4(av[c], hi, lo);
        *reinterpret_cast<float4*>(st + offs[c]) = hi;
        *reinterpret_cast<float4*>(st + TILE + offs[c]) = lo;
        if (b_ok) {
          split4(bv[c], hi, lo);
          *reinterpret_cast<float4*>(st + 2 * TILE + offs[c]) = hi;
          *reinterpret_cast<float4*>(st + 2 * TILE + TN_BT + offs[c]) = lo;
        }
      }
      if (n2) {   // feature rows follow the nt rows of the B tile (nt is a multiple of 8: the swizzle phase carries over)
        float4 hi, lo;
        split4(fv, hi, lo);
        *reinterpret_cast<float4*>(st + 2 * TILE + nt * 128 + foff) = hi;
        *reinterpret_cast<float4*>(st + 2 * TILE + TN_BT + nt * 128 + foff) = lo;
      }
      fence_proxy_async();
      mbar_arrive(&bar_full[cs]);
    }
    const int ngroups = (nchunks + TN_GROUP - 1) / TN_GROUP;
    if (nchunks > 0) mbar_wait(&bar_done, 0);
    for (; drained < ngroups; ++drained) drain(drained & 1);
    const bool row_ok = orow < kt, row_ok2 = orow < kt2;
    float* cp = nt > 0 ? segC + ((size_t)blockIdx.z * (sk1 - sk0) + (kg - sk0) + (row_ok ? orow : 0)) * a.N : nullptr;
    float* cp2 = n2 ? a.C2 + (size_t)blockIdx.z * a.c2_split + (size_t)(kg + (row_ok2 ? orow : 0)) * 32 : nullptr;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int c0 = half * 16 + 32 * i;
      if (c0 < ntot && (c0 < nt ? row_ok : row_ok2)) {
        float* o = c0 < nt ? cp + c0 : cp2 + (c0 - nt);
#pragma unroll
        for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[i][j], acc[i][j + 1], acc[i][j + 2], acc[i][j + 3]);
      }
    }
  } else if (warp == TN_W_MMA) {
    const uint32_t idesc = make_idesc(FMT_TF32, 128, max(ntot, 16), 0, 0);
    const uint32_t base = smem_u32(cv);
    for (int kc = 0; kc < nchunks; ++kc) {
      const int s = kc % TN_NC;
      const int g = kc / TN_GROUP, buf = g & 1, kg0 = kc % TN_GROUP;
      if (kg0 == 0 && g >= 2) {   // the converters have drained this accumulator's previous group (g - 2)
        mbar_wait(&bar_acc_free[buf], (uint32_t)((g / 2 - 1) & 1));
        tc_fence_after();
      }
      mbar_wait(&bar_full[s], (uint32_t)((kc / TN_NC) & 1));
      tc_fence_after();
      if (lane == 0) {
        const uint32_t st = base + s * TN_CV;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const uint32_t at = st + (p == 1 ? TILE : 0), bt = st + 2 * TILE + (p == 2 ? TN_BT : 0);
#pragma unroll
          for (int k = 0; k < KC / 8; ++k)
            umma<FMT_TF32>(tmem + buf * TN_ACC, make_desc(at + k * 32, 16, 1024, LAYOUT_SW128), make_desc(bt + k * 32, 16, 1024, LAYOUT_SW128),
                           idesc, (kg0 > 0 || p > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&bar_empty[s]);
        if (kc + 1 == nchunks) umma_commit(&bar_done);
      }
      __syncwarp();
    }
    tc_fence_before();
  } else {
    // ---- producer ----
    if (lane == 0 && nchunks > 0) {
      tmap_prefetch(&a.ta);
      if (sb >= 0) tmap_prefetch(&a.tb[sb]);
      if (n2) tmap_prefetch(&a.tf);
      const uint32_t bytes = (uint32_t)(TILE + (sb >= 0 ? a.N * 128 : 0) + (n2 ? TN_BOX : 0));
      for (int kc = 0; kc < nchunks; ++kc) {
        const int rs = kc % TN_NR;
        if (kc >= TN_NR) mbar_wait(&bar_rfree[rs], (uint32_t)((kc / TN_NR - 1) & 1));
        uint8_t* rw = raw + rs * KT_RAW;
        const long long tile = t0 + kc / 4;
        const int k0 = (kc & 3) * KC;
        mbar_arrive_expect_tx(&bar_raw[rs], bytes);
        const long long tq = tile * 4 + (k0 >> 5);      // (tile, row quarter)
        tma_2d(rw, &a.ta, 0, (int)(tq * a.Ktot + kg), &bar_raw[rs]);
        if (sb >= 0) tma_2d(rw + TILE, &a.tb[sb], 0, (int)(tq * a.N), &bar_raw[rs]);
        if (n2) tma_2d(rw + 2 * TILE, &a.tf, 0, (int)(tq * 32), &bar_raw[rs]);
      }
    }
  }
  __syncthreads();
  if (warp == TN_W_MMA) tmem_dealloc(tmem, 512);
}
}  // namespace

size_t gemm_nt_scratch_floats(int N, int K) { return (size_t)2 * ((N + 127) / 128 * 128) * ((K + KC - 1) / KC * KC); }

// C[M][N] = A[M][K] . Bt[N][K]^T for any M >= 1 (TMA zero-fills the rows of the last tile past M; they are not stored);
// `scratch` (gemm_nt_scratch_floats(N, K) floats) receives the hi / lo images of Bt.
int launch_gemm_nt_tma(const float* A, long long lda, const float* Bt, long long ldb, float* C, long long ldc, long long M, int N,
                       int K, float* scratch, cudaStream_t st) {
  REGT_CHECK(A && Bt && C && scratch && M >= 1 && N > 0 && N % 16 == 0 && K > 0 && K % 4 == 0 && ldc % 4 == 0 &&
                 ((uintptr_t)C % 16) == 0 && ((uintptr_t)scratch % 16) == 0,
             "gemm_nt_tma: bad operands (M=%lld N=%d K=%d)", M, N, K);
  const int Np = (N + 127) / 128 * 128, Kp = (K + KC - 1) / KC * KC, nchunks = Kp / KC;
  float* hi = scratch;
  float* lo = scratch + (size_t)Np * Kp;
  k_split_hilo<<<cdiv((long long)Np * Kp, 256), 256, 0, st>>>(Bt, ldb, N, K, Np, Kp, hi, lo);
  REGT_LAUNCHED("k_split_hilo", st);
  NtArgs a{};
  if (tmap_2d(&a.ta, A, K, M, lda, 128, "gemm_nt_tma(A)")) return -1;
  if (tmap_2d(&a.tbh, hi, Kp, Np, Kp, 128, "gemm_nt_tma(B hi)")) return -1;
  if (tmap_2d(&a.tbl, lo, Kp, Np, Kp, 128, "gemm_nt_tma(B lo)")) return -1;
  a.C = C; a.M = M; a.ldc = ldc; a.N = N; a.K = K;
  // shared memory holds the weights (parked when N, K <= 128, else streamed next to A) + raw fp32 A chunks only
  a.resident = (N <= 128 && nchunks * 2 * TILE + 2 * 2 * TILE <= SMEM_BUDGET) ? 1 : 0;
  const int fixed = a.resident ? nchunks * 2 * TILE : 0;
  const int stage_ts = a.resident ? TILE : 3 * TILE;
  a.ns = min(MAXS, (SMEM_BUDGET - fixed) / stage_ts);
  const long long ntiles = (long long)cdiv(M, 128) * cdiv(N, 128);
  const size_t smem_ts = (size_t)fixed + (size_t)a.ns * stage_ts + 1024;
  REGT_CUDA(cudaFuncSetAttribute(k_gemm_nt_tma_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ts));
  k_gemm_nt_tma_ts<<<(int)min(ntiles, (long long)sm_count()), NT_THREADS, smem_ts, st>>>(a);
  REGT_LAUNCHED("k_gemm_nt_tma_ts", st);
  return 0;
}

// One launch of the row contraction over several column segments of A (each K-tile of 128 columns belongs to one segment):
//   seg s: Cs[z][k1-k0][N] = partials of A[:, k0:k1]^T . B_s      (B_s = Bs[seg_b[s]], or none when seg_b[s] < 0)
//   and, for every segment, C2[z][k0:k1][32] = partials of A[:, k0:k1]^T . B2.
// Segment boundaries must be multiples of 128 unless there is a single segment.
int launch_gemm_tn_tma(const float* A, long long lda, long long M, int Ktot, int nseg, const int* seg_k0, const int* seg_b,
                       float* const* seg_C, const float* const* Bs, const long long* ldbs, int N, int splits, const float* B2,
                       long long ldb2, float* C2, long long c2_split, cudaStream_t st, int relu_b) {
  REGT_CHECK(A && nseg >= 1 && nseg <= 4 && Ktot % 32 == 0 && N % 32 == 0 && splits > 0 && M >= 1, "gemm_tn_tma: bad shape");
  REGT_CHECK(!B2 || (C2 && ldb2 % 4 == 0), "gemm_tn_tma: bad second operand");
  TnArgs a{};
  if (tmap_2d(&a.ta, A, Ktot, M, lda, 32, "gemm_tn_tma(A)")) return -1;
  bool any_b = false;
  for (int s = 0; s < nseg; ++s) {
    a.seg[s].k0 = seg_k0[s];
    a.seg[s].k1 = s + 1 < nseg ? seg_k0[s + 1] : Ktot;
    a.seg[s].b = seg_b[s];
    a.seg[s].C = seg_C[s];
    REGT_CHECK(nseg == 1 || a.seg[s].k0 % 128 == 0, "gemm_tn_tma: segment boundaries must be multiples of 128");
    REGT_CHECK(seg_b[s] < 2 && (seg_b[s] < 0 || (seg_C[s] && Bs[seg_b[s]])), "gemm_tn_tma: segment %d has no operand / output", s);
    any_b |= seg_b[s] >= 0;
  }
  for (int b = 0; b < 2; ++b) {
    bool used = false;
    for (int s = 0; s < nseg; ++s) used |= seg_b[s] == b;
    if (used && tmap_2d(&a.tb[b], Bs[b], N, M, ldbs[b], 32, "gemm_tn_tma(B)")) return -1;
  }
  REGT_CHECK(any_b || B2, "gemm_tn_tma: nothing to contract with");
  if (B2 && tmap_2d(&a.tf, B2, 32, M, ldb2, 32, "gemm_tn_tma(B2)")) return -1;
  a.nseg = nseg;
  a.C2 = C2;
  a.c2_split = c2_split > 0 ? c2_split : (long long)Ktot * 32;
  a.M = M;
  long long chunk = (M + splits - 1) / splits;
  a.chunk = (chunk + KC - 1) / KC * KC;
  a.N = any_b ? N : 0;
  a.N2 = B2 ? 32 : 0;
  a.relu_b = relu_b;
  const size_t smem = (size_t)TN_NR * TN_RAW + (size_t)TN_NC * TN_CV + 1024;
  REGT_CUDA(cudaFuncSetAttribute(k_gemm_tn_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_gemm_tn_tma<<<dim3(cdiv(Ktot, 128), max(1, cdiv(a.N, 128)), splits), TN_THREADS, smem, st>>>(a);
  REGT_LAUNCHED("k_gemm_tn_tma", st);
  return 0;
}

// the row contraction over transposed tiles (k_gemm_kt): AT [ntile][4][Ktot][32], BTs[b] [ntile][4][N][32], FT [ntile][4][32][32];
// segment boundaries are multiples of 128 columns except the end of the last segment with an operand (H = 64: [Dc | dhp])
int launch_gemm_kt(const float* AT, long long ntile, int Ktot, int nseg, const int* seg_k0, const int* seg_k1, const int* seg_b,
                   float* const* seg_C, const float* const* BTs, int N, int splits, const float* FT, float* C2, long long c2_split,
                   cudaStream_t st) {
  REGT_CHECK(AT && nseg >= 1 && nseg <= 4 && Ktot % 128 == 0 && N % 8 == 0 && N >= 16 && N <= 128 && splits > 0 && ntile > 0 && FT && C2,
             "gemm_kt: bad shape (Ktot=%d N=%d)", Ktot, N);
  REGT_CHECK(ntile * 4 * Ktot < (1ll << 31), "gemm_kt: tile count overflows the TMA coordinate");
  KtArgs a{};
  if (tmap_2d(&a.ta, AT, 32, ntile * 4 * Ktot, 32, 128, "gemm_kt(A^T)")) return -1;
  for (int s = 0; s < nseg; ++s) {
    a.seg[s].k0 = seg_k0[s];
    a.seg[s].k1 = seg_k1[s];
    a.seg[s].b = seg_b[s];
    a.seg[s].C = seg_C[s];
    REGT_CHECK(a.seg[s].k0 % 128 == 0, "gemm_kt: segment starts must be multiples of 128");
    REGT_CHECK(seg_b[s] < 2 && (seg_b[s] < 0 || (seg_C[s] && BTs[seg_b[s]])), "gemm_kt: segment %d has no operand / output", s);
  }
  for (int b = 0; b < 2; ++b) {
    bool used = false;
    for (int s = 0; s < nseg; ++s) used |= seg_b[s] == b;
    if (used && tmap_2d(&a.tb[b], BTs[b], 32, ntile * 4 * N, 32, N, "gemm_kt(B^T)")) return -1;
  }
  if (tmap_2d(&a.tf, FT, 32, ntile * 4 * 32, 32, 32, "gemm_kt(F^T)")) return -1;
  a.nseg = nseg;
  a.C2 = C2;
  a.c2_split = c2_split > 0 ? c2_split : (long long)Ktot * 32;
  a.ntile = ntile;
  a.tiles_per_split = (ntile + splits - 1) / splits;
  a.Ktot = Ktot; a.N = N; a.N2 = 32;
  const size_t smem = (size_t)TN_NR * KT_RAW + (size_t)TN_NC * TN_CV + 1024;
  REGT_CUDA(cudaFuncSetAttribute(k_gemm_kt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_gemm_kt<<<dim3(Ktot / 128, 1, splits), TN_THREADS, smem, st>>>(a);
  REGT_LAUNCHED("k_gemm_kt", st);
  return 0;
}

// the single-segment form of launch_gemm_tn_tma: Cp[z][K][N] = partials of A[:, :K]^T . B (no B when N == 0)
int launch_gemm_tn(const float* A, long long lda, const float* B, long long ldb, float* Cp, long long M, int K, int N, int splits,
                   cudaStream_t st, const float* B2, long long ldb2, float* Cp2, long long c2_split, int relu_b) {
  const int k0 = 0, sb = N > 0 ? 0 : -1;
  float* cs[1] = {Cp};
  const float* bs[2] = {B, nullptr};
  const long long lds[2] = {ldb, 0};
  return launch_gemm_tn_tma(A, lda, M, K, 1, &k0, &sb, cs, bs, lds, N, splits, B2, ldb2, Cp2, c2_split, st, relu_b);
}

}  // namespace regt

// debug entry points (not part of the reference-facing ABI): tests/test_gpu_gemm.py
extern "C" int regt_debug_gemm_nt_tma(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc, int64_t M,
                                      int32_t N, int32_t K, float* scratch, regt_stream_t stream) {
  return regt::launch_gemm_nt_tma(A, lda, Bt, ldb, C, ldc, M, N, K, scratch, (cudaStream_t)stream);
}
extern "C" int regt_debug_gemm_tn_tma(const float* A, int64_t lda, const float* B, int64_t ldb, float* Cp, int64_t M, int32_t K,
                                      int32_t N, int32_t splits, const float* B2, int64_t ldb2, float* Cp2, regt_stream_t stream) {
  return regt::launch_gemm_tn(A, lda, B, ldb, Cp, M, K, N, splits, (cudaStream_t)stream, B2, ldb2, Cp2, 0, 0);
}
// four-segment form used by the cell backward: A = D [M][4H]; segments z|r (B = h), h~ (B = hR), h_pre (B2 only)
extern "C" int regt_debug_gemm_tn_multi(const float* A, int64_t lda, int64_t M, int32_t H, const float* B0, const float* B1,
                                        float* C0, float* C1, int32_t splits, const float* B2, float* C2, regt_stream_t stream) {
  const int k0[3] = {0, 2 * H, 3 * H}, sb[3] = {0, 1, -1};
  float* cs[3] = {C0, C1, nullptr};
  const float* bs[2] = {B0, B1};
  const long long lds[2] = {H, H};
  return regt::launch_gemm_tn_tma(A, lda, M, 4 * H, 3, k0, sb, cs, bs, lds, H, splits, B2, 32, C2, 0, (cudaStream_t)stream, 0);
}
// the transposed-tile form used by the fused cell backward: AT [ntile][4][4H][32]; B0T, B1T [ntile][4][H][32]; FT [ntile][4][32][32]
extern "C" int regt_debug_gemm_kt(const float* AT, int64_t ntile, int32_t H, const float* B0T, const float* B1T, const float* FT,
                                  float* C0, float* C1, float* C2, int32_t splits, regt_stream_t stream) {
  int k0[3], k1[3], sb[3], ns;
  float* cs[3];
  if (H == 128) {
    ns = 3;
    k0[0] = 0; k1[0] = 256; sb[0] = 0; cs[0] = C0;
    k0[1] = 256; k1[1] = 384; sb[1] = 1; cs[1] = C1;
    k0[2] = 384; k1[2] = 512; sb[2] = -1; cs[2] = nullptr;
  } else {
    ns = 2;
    k0[0] = 0; k1[0] = 128; sb[0] = 0; cs[0] = C0;
    k0[1] = 128; k1[1] = 192; sb[1] = 1; cs[1] = C1;
  }
  const float* bs[2] = {B0T, B1T};
  return regt::launch_gemm_kt(AT, ntile, 4 * H, ns, k0, k1, sb, cs, bs, H, splits, FT, C2, 0, (cudaStream_t)stream);
}
