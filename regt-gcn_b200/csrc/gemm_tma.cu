// TMA-fed 3xTF32 GEMMs, and their single-pass bf16 forms.
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
//
// Each pipeline is written once: gemm_nt<GemmKind> for both precisions of gemm_nt, and gemm_rows<Policy> for the three row
// contractions (k_gemm_tn_tma, k_gemm_kt, k_gemm_tn_bf16), whose operand policies supply only the boxes of a chunk, its
// conversion and its MMAs.  The __global__ kernels are thin wrappers that keep their names for the profiles.
#include <cuda.h>   // CUtensorMap and its enums only: the encoder is fetched through the runtime (no libcuda link)

#include "cell_tc.cuh"

namespace regt {
using namespace tc;

namespace {
constexpr int KC = 32;               // contraction chunk: 32 fp32 = one 128-byte swizzle row
constexpr int KB = 64;               // bf16 contraction chunk: one 128-byte swizzle row
constexpr int TILE = 128 * 128;      // [128 rows][128 B] operand tile
constexpr int MAXS = 6;              // pipeline stages (upper bound)
constexpr int SMEM_BUDGET = 227 * 1024 - 1024;   // dynamic shared memory minus the 1024-byte alignment slack

__device__ __forceinline__ void split4(const float4 v, float4& hi, float4& lo) {
  hi.x = __uint_as_float(tf32_rn(v.x)); hi.y = __uint_as_float(tf32_rn(v.y));
  hi.z = __uint_as_float(tf32_rn(v.z)); hi.w = __uint_as_float(tf32_rn(v.w));
  lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
}
__device__ __forceinline__ uint4 pack8_bf16(const float4 u, const float4 v) {
  return make_uint4(pack_bf16(u.x, u.y), pack_bf16(u.z, u.w), pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
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
// A raw stage is refilled by TMA once every converter thread has arrived on its `free` barrier, and an mbarrier arrive does
// NOT wait for this thread's earlier shared-memory loads to return (observed on B200: the tail loads of a warp read the NEXT
// chunk's bytes).  A branch on the loaded values (`dep`: an OR of words of them) forces their completion before the arrive.
__device__ __forceinline__ void release_stage(uint32_t dep, uint64_t* free_bar) {
  if (dep == 0x7FC0DEADu) __nanosleep(1);
  mbar_arrive(free_bar);
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
// T = float or __nv_bfloat16: [rows][cols] window of a row-major array with pitch ld (elements); boxes of box_rows x one
// 128-byte swizzle row (32 fp32 or 64 bf16), out-of-range elements read as zero
template <class T>
int tmap_2d(CUtensorMap* m, const T* base, long long cols, long long rows, long long ld, int box_rows, const char* who) {
  static_assert(sizeof(T) == 4 || sizeof(T) == 2, "fp32 or bf16 elements");
  EncodeFn enc = encoder();
  REGT_CHECK(enc != nullptr, "%s: cuTensorMapEncodeTiled is not available from this driver", who);
  REGT_CHECK(((uintptr_t)base % 16 == 0) && ld % (long long)(16 / sizeof(T)) == 0,"%s: TMA operands need 16-byte aligned base and pitch", who);
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(T)};
  cuuint32_t box[2] = {128 / sizeof(T), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType type = sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const CUresult r = enc(m, type, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  REGT_CHECK(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed (%d) cols=%lld rows=%lld ld=%lld", who, (int)r, cols, rows, ld);
  return 0;
}

// ------------------------------------------------------------------------------------------
// dense images of a weight operand, zero-padded to [Np][Kp]: tf32 hi[n][k] = tf32(B[n][k]), lo = B - hi; or bf16(B[n][k])
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
__global__ void k_pack_bf16(const float* __restrict__ B, long long ldb, int N, int K, int Np, int Kp, __nv_bfloat16* __restrict__ img) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)Np * Kp) return;
  const int n = (int)(i / Kp), k = (int)(i - (long long)n * Kp);
  img[i] = __float2bfloat16_rn((n < N && k < K) ? __ldg(B + (size_t)n * ldb + k) : 0.f);
}

// ------------------------------------------------------------------------------------------
// Single-pass bf16 forms of gemm_nt and gemm_tn (precision bf16 on the GEMM-by-GEMM cell of cell_g.cu).  The operands
// still arrive by TMA as fp32 and C stays fp32; the converters round each operand to bf16 once (round to nearest even)
// instead of splitting it into tf32 hi / lo, and every K step is ONE kind::f16 MMA with fp32 accumulation in TMEM.
// A 128-byte swizzle row holds 64 bf16 but only 32 fp32, so a chunk is KB = 64 contraction elements, fed by two 32-wide
// fp32 boxes:
//   gemm_nt: A chunk = two [128 rows][32 k] fp32 boxes -> one K-major SW128 bf16 tile [128 rows][64 k] (the layout of
//            umma_selftest variant 0); the weight operand is packed ONCE per call into a dense bf16 image (k_pack_bf16)
//            whose [128][64] TMA boxes land in that same layout, parked in shared memory (N <= 128, K <= 384) or streamed.
//            A is read from SHARED memory, not TMEM: a converted tile is 16 KB (half the tf32 hi | lo pair), so four of
//            them beside the raw stages still leave 3-4 stages = 96-128 KB of loads in flight (the TS kernel keeps 96 KB),
//            and both operands then use the one bf16 layout umma_selftest pins; no test here pins the TMEM layout of a
//            16-bit A operand.
//   gemm_tn: raw boxes [64 rows][32 cols] fp32 and NO transpose: the contraction runs over the rows of the boxes, so each
//            row is converted in place of position into MN-major SW128 bf16 tiles [cols / 64][64 rows][128 B] (the
//            layout of umma_selftest variant 2; one 16-byte store per two 16-byte loads, where the tf32 converters issue
//            eight 4-byte transposing stores).  The 32 columns of B2 follow the B columns of the tile as its last box.
// ------------------------------------------------------------------------------------------

// ------------------------------------------------------------------------------------------
// gemm_nt.  tf32x3: A operand through TMEM ("TS" MMAs).  With the weight operand parked in shared memory (128 KB at
// N = K = 128) a version that kept [A hi | A lo] in shared memory had room for 3 stages = 48 KB of TMA loads in flight and
// ran at 55 % of the HBM bandwidth (measured in round 1, since removed).  Here the converters write hi / lo straight into
// TMEM (tcgen05.st, 4 slots x 64 columns next to the two 128-column accumulators), the MMAs read A from there, and shared
// memory holds only RAW fp32 chunks: 6 stages x 16 KB in flight (H = 128: 1.11 -> 0.88 ms, 4.5 TB/s = 68 % of the
// measured HBM peak).  Streamed weights (N or K > 128): a stage is [raw A | B hi | B lo] = 48 KB, four of them.
// bf16: a stage is [two raw A boxes ( | bf16 B tile when the weights stream)], the converted A tiles sit in NB_SLOTS
// shared-memory slots after the parked weights.
// ------------------------------------------------------------------------------------------
struct NtArgs {
  CUtensorMap ta, tb[2];      // A [M][K] fp32; Bt: tf32 hi / lo images [Np][Kp] (Tf32x3), or its bf16 image in tb[0] (Bf16)
  float* C;
  long long M, ldc;
  int N, K;
  int resident;               // the weight images parked in shared memory for the whole kernel
  int ns;                     // pipeline stages
};
constexpr int NT_CONV = 256;                    // converter threads (warps 0-7)
constexpr int NT_W_TMA = NT_CONV / 32;          // producer warp
constexpr int NT_W_MMA = NT_W_TMA + 1;          // MMA issuer (owns the TMEM allocation)
constexpr int NT_W_EPI = NT_W_MMA + 1;          // 4 epilogue warps
constexpr int NT_THREADS = (NT_W_EPI + 4) * 32;
constexpr int TS_SLOTS = 4;      // tf32x3: A (hi | lo) slots in TMEM, 64 columns each, after the two accumulators
constexpr int NB_SLOTS = 4;      // bf16: converted A tiles in shared memory

// a chunk of gemm_nt: contraction elements, raw fp32 A bytes, weight bytes (tf32 hi | lo tiles or one bf16 tile) and the
// shared memory of the converted A slots
struct NtGeom {
  int ck, raw_a, wt, aslots;
};
__host__ __device__ constexpr NtGeom nt_geom(GemmKind g) {
  return g == GemmKind::Bf16 ? NtGeom{KB, 2 * TILE, TILE, NB_SLOTS * TILE} : NtGeom{KC, TILE, 2 * TILE, 0};
}

template <GemmKind G>
__device__ __forceinline__ void gemm_nt(const NtArgs& a) {
  constexpr bool BF = G == GemmKind::Bf16;
  constexpr NtGeom g = nt_geom(G);
  constexpr int SLOTS = BF ? NB_SLOTS : TS_SLOTS;
  constexpr int NW = BF ? 1 : 2;                    // weight images: bf16, or tf32 hi and lo
  constexpr uint32_t TMEM_COLS = BF ? 256 : 512;    // the two accumulators (+ the A slots of tf32x3)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_tma[MAXS], bar_rfree[MAXS], bar_afull[SLOTS], bar_afree[SLOTS], bar_b, bar_acc_full[2], bar_acc_free[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ns = a.ns;
  const int nchunks = (a.K + g.ck - 1) / g.ck;
  const int ntn = (a.N + 127) / 128;
  const long long ntiles = ((a.M + 127) / 128) * ntn;
  const int stage_bytes = g.raw_a + (a.resident ? 0 : g.wt);   // raw fp32 A chunk ( | the weight tiles when they stream)
  uint8_t* bres = sm;
  uint8_t* aslot = sm + (a.resident ? nchunks * g.wt : 0);
  uint8_t* stages = aslot + g.aslots;
  if (tid == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(&bar_tma[s], 1);
      mbar_init(&bar_rfree[s], a.resident ? NT_CONV : NT_CONV + 1);   // streamed weights: + the commit of the MMAs that read them
    }
    for (int s = 0; s < SLOTS; ++s) {
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
  if (warp == NT_W_MMA) tmem_alloc(&tmem_base_s, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t tmem_a = tmem + 256;              // tf32x3 slot s: hi at columns 64 s .. +31, lo at 64 s + 32 .. +63

  if (warp < NT_W_TMA) {
    // ---- converters: thread = (row of the tile, half of the chunk); the two warps of a TMEM lane quarter take one half
    //      each.  tf32x3: half = 16 of the chunk's 32 k; bf16: half = raw box `half` = k 32 half .. + 31, two 16-byte raw
    //      pieces make one 16-byte piece of the bf16 row.  Raw rows are 128-byte swizzled: the 8 lanes of a quarter-warp
    //      read 8 different banks groups.
    const int q = warp & 3, half = warp >> 2;
    const int r = q * 32 + lane, sw = r & 7;
    const uint32_t tl = tmem_a + ((uint32_t)(q * 32) << 16) + 16 * half;
    long long gc = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      for (int kc = 0; kc < nchunks; ++kc, ++gc) {
        const int s = (int)(gc % ns), sl = (int)(gc % SLOTS);
        mbar_wait(&bar_tma[s], (uint32_t)((gc / ns) & 1));
        const uint8_t* rw = stages + (size_t)s * stage_bytes + r * 128;
        if constexpr (BF) {
          uint4 p[4] = {make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u)};
          if (kc * KB + 32 * half < a.K) {   // the box was loaded (a box wholly past K is not)
#pragma unroll
            for (int c = 0; c < 4; ++c)
              p[c] = pack8_bf16(*reinterpret_cast<const float4*>(rw + half * TILE + (((2 * c) ^ sw) << 4)),
                                *reinterpret_cast<const float4*>(rw + half * TILE + (((2 * c + 1) ^ sw) << 4)));
          }
          release_stage(p[0].x | p[1].x | p[2].x | p[3].x, &bar_rfree[s]);
          if (gc >= SLOTS) mbar_wait(&bar_afree[sl], (uint32_t)((gc / SLOTS - 1) & 1));
          uint8_t* dst = aslot + (size_t)sl * TILE + r * 128;
#pragma unroll
          for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(dst + (((4 * half + c) ^ sw) << 4)) = p[c];
          fence_proxy_async();
        } else {
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 v = *reinterpret_cast<const float4*>(rw + (((half * 4 + c) ^ sw) << 4));
            float4 h, l;
            split4(v, h, l);
            hi[4 * c] = __float_as_uint(h.x); hi[4 * c + 1] = __float_as_uint(h.y); hi[4 * c + 2] = __float_as_uint(h.z); hi[4 * c + 3] = __float_as_uint(h.w);
            lo[4 * c] = __float_as_uint(l.x); lo[4 * c + 1] = __float_as_uint(l.y); lo[4 * c + 2] = __float_as_uint(l.z); lo[4 * c + 3] = __float_as_uint(l.w);
          }
          release_stage(hi[0] | hi[4] | hi[8] | hi[12], &bar_rfree[s]);
          if (gc >= SLOTS) {
            mbar_wait(&bar_afree[sl], (uint32_t)((gc / SLOTS - 1) & 1));
            tc_fence_after();
          }
          tmem_st16(tl + 64 * sl, hi);
          tmem_st16(tl + 64 * sl + 32, lo);
          tmem_st_wait();
          tc_fence_before();
        }
        mbar_arrive(&bar_afull[sl]);
      }
    }
  } else if (warp == NT_W_TMA) {
    if (lane == 0) {
      tmap_prefetch(&a.ta);
#pragma unroll
      for (int w = 0; w < NW; ++w) tmap_prefetch(&a.tb[w]);
      if (a.resident) {
        mbar_arrive_expect_tx(&bar_b, (uint32_t)(nchunks * g.wt));
        for (int kc = 0; kc < nchunks; ++kc)
#pragma unroll
          for (int w = 0; w < NW; ++w) tma_2d(bres + (size_t)kc * g.wt + w * TILE, &a.tb[w], kc * g.ck, 0, &bar_b);
      }
      long long gc = 0;
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int m0 = (int)((tile / ntn) * 128), n0 = (int)(tile % ntn) * 128;
        for (int kc = 0; kc < nchunks; ++kc, ++gc) {
          const int s = (int)(gc % ns);
          if (gc >= ns) mbar_wait(&bar_rfree[s], (uint32_t)((gc / ns - 1) & 1));
          uint8_t* st = stages + (size_t)s * stage_bytes;
          const bool second = BF && kc * KB + 32 < a.K;   // bf16: the chunk's second A box, unless it lies wholly past K
          mbar_arrive_expect_tx(&bar_tma[s], (uint32_t)(stage_bytes - (BF && !second ? TILE : 0)));
          tma_2d(st, &a.ta, kc * g.ck, m0, &bar_tma[s]);
          if (second) tma_2d(st + TILE, &a.ta, kc * KB + 32, m0, &bar_tma[s]);
          if (!a.resident)
#pragma unroll
            for (int w = 0; w < NW; ++w) tma_2d(st + g.raw_a + w * TILE, &a.tb[w], kc * g.ck, n0, &bar_tma[s]);
        }
      }
    }
  } else if (warp == NT_W_MMA) {
    const uint32_t bres0 = smem_u32(bres), aslot0 = smem_u32(aslot), stage0 = smem_u32(stages);
    if (a.resident) mbar_wait(&bar_b, 0);
    long long gc = 0, li = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++li) {
      const int nt = min(128, a.N - (int)(tile % ntn) * 128);
      const uint32_t idesc = make_idesc(BF ? FMT_BF16 : FMT_TF32, 128, nt, 0, 0);
      const int buf = (int)(li & 1);
      if (li >= 2) {
        mbar_wait(&bar_acc_free[buf], (uint32_t)((li / 2 - 1) & 1));
        tc_fence_after();
      }
      for (int kc = 0; kc < nchunks; ++kc, ++gc) {
        const int sl = (int)(gc % SLOTS);
        mbar_wait(&bar_afull[sl], (uint32_t)((gc / SLOTS) & 1));
        tc_fence_after();
        if (lane == 0) {
          const int s = (int)(gc % ns);
          const uint32_t bt = a.resident ? bres0 + kc * g.wt : stage0 + s * stage_bytes + g.raw_a;
          if constexpr (BF) {
            const uint32_t at = aslot0 + sl * TILE;
#pragma unroll
            for (int k = 0; k < KB / 16; ++k)
              umma<FMT_BF16>(tmem + buf * 128, make_desc(at + k * 32, 16, 1024, LAYOUT_SW128), make_desc(bt + k * 32, 16, 1024, LAYOUT_SW128),
                             idesc, (kc > 0 || k > 0) ? 1u : 0u);
          } else {
            const uint32_t ah = tmem_a + 64 * sl, al = ah + 32;
#pragma unroll
            for (int p = 0; p < 3; ++p) {   // hi*hi, lo*hi, hi*lo
              const uint32_t ap = (p == 1) ? al : ah, bp = bt + (p == 2 ? TILE : 0);
#pragma unroll
              for (int k = 0; k < KC / 8; ++k)
                umma_ts_tf32(tmem + buf * 128, ap + 8 * k, make_desc(bp + k * 32, 16, 1024, LAYOUT_SW128), idesc,
                             (kc > 0 || p > 0 || k > 0) ? 1u : 0u);
            }
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
  if (warp == NT_W_MMA) tmem_dealloc(tmem, TMEM_COLS);
}

__global__ void __launch_bounds__(NT_THREADS, 1) k_gemm_nt_tma_ts(const __grid_constant__ NtArgs a) { gemm_nt<GemmKind::Tf32x3>(a); }
__global__ void __launch_bounds__(NT_THREADS, 1) k_gemm_nt_bf16(const __grid_constant__ NtArgs a) { gemm_nt<GemmKind::Bf16>(a); }

// ------------------------------------------------------------------------------------------
// the row contraction (gemm_tn, and gemm_kt below)
// ------------------------------------------------------------------------------------------
struct TnSeg {
  int k0, k1;   // columns [k0, k1) of A
  int b;        // B operand of this segment: index into tb[], or -1 (only the B2 plane)
  float* C;     // [split][k1 - k0][N]
};
struct TnArgs {
  CUtensorMap ta, tb[2], tf;   // A, B operands, B2: row-major [M][Ktot], [M][N], [M][32], or gemm_kt's transposed tiles
  TnSeg seg[4];
  int nseg;
  float* C2;                   // [split][Ktot][32] (stride c2_split between splits)
  long long c2_split;
  long long M, chunk;          // rows contracted over; rows per split (a multiple of the rows of a chunk)
  int Ktot, N, N2;
  int relu_b;                  // the B operands are read through max(., 0)
};
// this CTA's output tile
struct TnTile {
  int kg, n0;   // first column of A and of the B operand
  int kt;       // output rows that belong to the segment's C
  int sb;       // B operand of the segment, or -1
  int nt, n2;   // columns from the B operand; + the 32 feature columns on N tile 0
};
constexpr int TN_CONV = 256;                  // converter / epilogue threads (warps 0-7)
constexpr int TN_W_MMA = TN_CONV / 32;
constexpr int TN_W_TMA = TN_W_MMA + 1;
constexpr int TN_THREADS = (TN_W_TMA + 1) * 32;
constexpr int TN_NR = 2, TN_NC = 2;           // raw (TMA) stages, converted (MMA operand) stages
constexpr int TN_BOX = 32 * 128;              // one [32 rows][32 cols] fp32 box
constexpr int TN_BT = (128 + 32) * 128;       // converted B tile with the 32 extra feature rows
constexpr int TN_CV = 2 * TILE + 2 * TN_BT;   // A hi | A lo | B hi | B lo
// The tensor core's fp32 accumulation is not round-to-nearest: its error grows linearly with the number of MMAs
// chained into one accumulator (measured ~2e-8 relative per MMA).  A row contraction chains 12 MMAs per chunk over up to
// 10^5 rows, so the TMEM accumulator is drained into fp32 registers (round-to-nearest adds) every TN_GROUP chunks; two
// accumulators alternate so the drain of group g runs under the MMAs of group g + 1.
constexpr int TN_GROUP = 8;
constexpr int TN_ACC = 256;                   // TMEM column stride between the two accumulators (each 128 + 32 feature columns wide)

// ---- operand policies.  A policy gives the rows of a chunk (ROWS), its raw and converted stage sizes (RAW, CV), the MMA
//      format and majors (FMT, MN), the producer's boxes of the chunk at row `row` and their byte count, and a converter
//      thread: load() reads the thread's part of a raw stage and returns the dependence word of release_stage, store()
//      writes it as MMA operand; mma() issues one chunk's MMAs into an accumulator.

// the boxes of a chunk of row-major operands: A columns kg.., B columns n0.. of operand sb, the B2 plane
template <int BOX>
__device__ __forceinline__ uint32_t row_bytes(const TnTile& t) {
  return (uint32_t)((t.kt / 32 + t.nt / 32 + (t.n2 ? 1 : 0)) * BOX);
}
template <int BOX>
__device__ __forceinline__ void row_boxes(uint8_t* rw, const TnArgs& a, const TnTile& t, int row, uint64_t* bar) {
  for (int b = 0; b < t.kt / 32; ++b) tma_2d(rw + b * BOX, &a.ta, t.kg + b * 32, row, bar);
  for (int b = 0; b < t.nt / 32; ++b) tma_2d(rw + (4 + b) * BOX, &a.tb[t.sb], t.n0 + b * 32, row, bar);
  if (t.n2) tma_2d(rw + 8 * BOX, &a.tf, 0, row, bar);
}
// the 3xTF32 MMAs of a chunk over a converted stage [A hi | A lo | B hi | B lo] (K-major SW128): hi*hi, lo*hi, hi*lo
__device__ __forceinline__ void mma_tf32x3(uint32_t d, uint32_t st, uint32_t idesc, bool acc) {
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    const uint32_t at = st + (p == 1 ? TILE : 0), bt = st + 2 * TILE + (p == 2 ? TN_BT : 0);
#pragma unroll
    for (int k = 0; k < KC / 8; ++k)
      umma<FMT_TF32>(d, make_desc(at + k * 32, 16, 1024, LAYOUT_SW128), make_desc(bt + k * 32, 16, 1024, LAYOUT_SW128), idesc,
                     (acc || p > 0 || k > 0) ? 1u : 0u);
  }
}

// row-major fp32 operands, tf32x3: raw [32 rows][32 cols] boxes (A: 4, B: 4, B2: 1) transposed into K-major hi / lo tiles
struct TnTf32 {
  static constexpr int ROWS = KC, BOX = TN_BOX, RAW = 9 * BOX, CV = TN_CV, FMT = FMT_TF32, MN = 0;
  __device__ static uint32_t bytes(const TnArgs&, const TnTile& t) { return row_bytes<BOX>(t); }
  __device__ static void boxes(uint8_t* rw, const TnArgs& a, const TnTile& t, int row, uint64_t* bar) { row_boxes<BOX>(rw, a, t, row, bar); }
  __device__ static void mma(uint32_t d, uint32_t st, uint32_t idesc, bool acc) { mma_tf32x3(d, st, idesc, acc); }

  // converter: warp (w & 3) owns column block w & 3 of A and of B, its half w >> 2 four float4s of that block; lane = row
  // of the chunk.  The raw boxes are 128-byte swizzled, so the eight lanes of a quarter-warp read eight different 16-byte
  // columns; the transposed 4-byte stores of one (c, e) hit 32 different banks.
  int warp, lane, blk, half, nt, n2;
  bool a_ok, b_ok, relu;
  float4 av[4], bv[4], fv;
  __device__ TnTf32(const TnArgs& a, const TnTile& t, int tid)
      : warp(tid >> 5), lane(tid & 31), blk(warp & 3), half(warp >> 2), nt(t.nt), n2(t.n2), a_ok(blk < t.kt / 32),
        b_ok(blk < t.nt / 32), relu(a.relu_b != 0) {}
  __device__ uint32_t load(const uint8_t* rw) {
    fv = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const uint32_t off = (uint32_t)(lane * 128 + (((half * 4 + c) ^ (lane & 7)) << 4));
      av[c] = a_ok ? *reinterpret_cast<const float4*>(rw + blk * BOX + off) : make_float4(0.f, 0.f, 0.f, 0.f);
      bv[c] = b_ok ? *reinterpret_cast<const float4*>(rw + (4 + blk) * BOX + off) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (relu) {
#pragma unroll
      for (int c = 0; c < 4; ++c) bv[c] = make_float4(fmaxf(bv[c].x, 0.f), fmaxf(bv[c].y, 0.f), fmaxf(bv[c].z, 0.f), fmaxf(bv[c].w, 0.f));
    }
    if (n2) fv = *reinterpret_cast<const float4*>(rw + 8 * BOX + lane * 128 + ((warp ^ (lane & 7)) << 4));
    return __float_as_uint(av[0].x) | __float_as_uint(av[1].x) | __float_as_uint(av[2].x) | __float_as_uint(av[3].x) |
           __float_as_uint(bv[0].x) | __float_as_uint(bv[1].x) | __float_as_uint(bv[2].x) | __float_as_uint(bv[3].x) | __float_as_uint(fv.x);
  }
  __device__ void store(uint8_t* st) const {
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
  }
};

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
// (a chunk = one row quarter of a tile: the 32 rows a warp of the producing kernel owns; row r of the contraction is row
// r % 128 of tile r / 128)
// ------------------------------------------------------------------------------------------
struct Kt {
  static constexpr int ROWS = KC, BOX = TN_BOX, RAW = 2 * TILE + BOX, CV = TN_CV, FMT = FMT_TF32, MN = 0;   // raw: A^T | B^T | F^T
  __device__ static uint32_t bytes(const TnArgs&, const TnTile& t) { return (uint32_t)(TILE + t.nt * 128 + (t.n2 ? BOX : 0)); }
  __device__ static void boxes(uint8_t* rw, const TnArgs& a, const TnTile& t, int row, uint64_t* bar) {
    const int tq = row / KC;   // (tile, row quarter)
    tma_2d(rw, &a.ta, 0, tq * a.Ktot + t.kg, bar);
    if (t.sb >= 0) tma_2d(rw + TILE, &a.tb[t.sb], 0, tq * a.N, bar);
    if (t.n2) tma_2d(rw + 2 * TILE, &a.tf, 0, tq * 32, bar);
  }
  __device__ static void mma(uint32_t d, uint32_t st, uint32_t idesc, bool acc) { mma_tf32x3(d, st, idesc, acc); }

  // converter: thread = (row of the A^T / B^T tile, four of its eight 16-byte pieces); feature tile: (row tid / 8, piece tid % 8)
  int nt, n2;
  bool b_ok;
  uint32_t offs[4], foff;
  float4 av[4], bv[4], fv;
  __device__ Kt(const TnArgs&, const TnTile& t, int tid) : nt(t.nt), n2(t.n2) {
    const int warp = tid >> 5, row = (warp & 3) * 32 + (tid & 31), half = warp >> 2;
    const int frow = tid >> 3, fpc = tid & 7;
    b_ok = row < nt;
#pragma unroll
    for (int c = 0; c < 4; ++c) offs[c] = (uint32_t)(row * 128 + (((half * 4 + c) ^ (row & 7)) << 4));
    foff = (uint32_t)(frow * 128 + ((fpc ^ (frow & 7)) << 4));
  }
  __device__ uint32_t load(const uint8_t* rw) {
    fv = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      av[c] = *reinterpret_cast<const float4*>(rw + offs[c]);
      bv[c] = b_ok ? *reinterpret_cast<const float4*>(rw + TILE + offs[c]) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (n2) fv = *reinterpret_cast<const float4*>(rw + 2 * TILE + foff);
    return __float_as_uint(av[0].x) | __float_as_uint(av[1].x) | __float_as_uint(av[2].x) | __float_as_uint(av[3].x) |
           __float_as_uint(bv[0].x) | __float_as_uint(bv[1].x) | __float_as_uint(bv[2].x) | __float_as_uint(bv[3].x) | __float_as_uint(fv.x);
  }
  __device__ void store(uint8_t* st) const {
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
  }
};

// row-major fp32 operands, single-pass bf16 (see above): raw [64 rows][32 cols] boxes converted into MN-major tiles
constexpr int TB_BOX = KB * 128;              // one [64 rows][32 cols] fp32 box
constexpr int TB_BLK = KB * 128;              // one MN-major bf16 block: 64 columns x 64 rows
constexpr int TB_AT = 2 * TB_BLK;             // converted A tile: 128 columns
constexpr int TB_CV = TB_AT + 3 * TB_BLK;     // A | B tile of 128 + 32 feature columns

// raw box b (columns 32 b .. 32 b + 31 of its operand), quarter p of row `row`, converted: 8 bf16 for byte 16 p of the row
__device__ __forceinline__ uint4 tb_piece(const uint8_t* rw_row, int b, int p, int sw, bool relu) {
  const uint8_t* src = rw_row + b * TB_BOX;
  float4 u = *reinterpret_cast<const float4*>(src + (((2 * p) ^ sw) << 4));
  float4 v = *reinterpret_cast<const float4*>(src + (((2 * p + 1) ^ sw) << 4));
  if (relu) {
    u = make_float4(fmaxf(u.x, 0.f), fmaxf(u.y, 0.f), fmaxf(u.z, 0.f), fmaxf(u.w, 0.f));
    v = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
  }
  return pack8_bf16(u, v);
}
// byte offset of column box b, quarter p of row `row` in an MN-major SW128 bf16 tile [blocks of 64 columns][64 rows][128 B]
__device__ __forceinline__ uint32_t tb_off(int b, int p, int row) {
  return (uint32_t)((b >> 1) * TB_BLK + row * 128 + ((((b & 1) * 4 + p) ^ (row & 7)) << 4));
}

struct TnBf16 {
  static constexpr int ROWS = KB, BOX = TB_BOX, RAW = 9 * BOX, CV = TB_CV, FMT = FMT_BF16, MN = 1;
  __device__ static uint32_t bytes(const TnArgs&, const TnTile& t) { return row_bytes<BOX>(t); }
  __device__ static void boxes(uint8_t* rw, const TnArgs& a, const TnTile& t, int row, uint64_t* bar) { row_boxes<BOX>(rw, a, t, row, bar); }
  __device__ static void mma(uint32_t d, uint32_t st, uint32_t idesc, bool acc) {
    const uint32_t at = st, bt = at + TB_AT;
    // MN-major: LBO = stride of the 64-column blocks, SBO = stride of 8-row groups; a K step is 16 rows = 2 KB
#pragma unroll
    for (int k = 0; k < KB / 16; ++k)
      umma<FMT_BF16>(d, make_desc(at + k * 2048, TB_BLK, 1024, LAYOUT_SW128), make_desc(bt + k * 2048, TB_BLK, 1024, LAYOUT_SW128), idesc,
                     (acc || k > 0) ? 1u : 0u);
  }

  // converter: thread = (row of the chunk tid % 64, 16-byte quarter tid / 64 of every box's bf16 row); the feature box,
  // when present, is box bblk of B
  int row, p, sw, ablk, bblk, n2;
  bool relu;
  uint4 av[4], bv[5];
  __device__ TnBf16(const TnArgs& a, const TnTile& t, int tid)
      : row(tid & 63), p(tid >> 6), sw(row & 7), ablk(t.kt / 32), bblk(t.nt / 32), n2(t.n2), relu(a.relu_b != 0) {}
  __device__ uint32_t load(const uint8_t* rw) {
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    rw += row * 128;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      av[b] = b < ablk ? tb_piece(rw, b, p, sw, false) : zero;
      bv[b] = b < bblk ? tb_piece(rw, 4 + b, p, sw, relu) : zero;
    }
    bv[4] = n2 ? tb_piece(rw, 8, p, sw, false) : zero;
    return av[0].x | av[1].x | av[2].x | av[3].x | bv[0].x | bv[1].x | bv[2].x | bv[3].x | bv[4].x;
  }
  __device__ void store(uint8_t* st) const {
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      *reinterpret_cast<uint4*>(st + tb_off(b, p, row)) = av[b];
      if (b < bblk) *reinterpret_cast<uint4*>(st + TB_AT + tb_off(b, p, row)) = bv[b];
    }
    if (n2) *reinterpret_cast<uint4*>(st + TB_AT + tb_off(bblk, p, row)) = bv[4];
  }
};
static_assert(TN_NR * TnTf32::RAW + TN_NC * TnTf32::CV <= SMEM_BUDGET, "gemm_tn stages exceed shared memory");
static_assert(TN_NR * TnBf16::RAW + TN_NC * TnBf16::CV <= SMEM_BUDGET, "bf16 gemm_tn stages exceed shared memory");

template <class P>
__device__ __forceinline__ void gemm_rows(const TnArgs& a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_raw[TN_NR], bar_rfree[TN_NR], bar_full[TN_NC], bar_empty[TN_NC], bar_done, bar_acc_free[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  TnTile t;
  t.kg = blockIdx.x * 128;
  int si = 0;
  for (int s = 1; s < a.nseg; ++s)
    if (t.kg >= a.seg[s].k0) si = s;
  const int sk0 = a.seg[si].k0, sk1 = a.seg[si].k1;
  float* segC = a.seg[si].C;
  t.sb = a.seg[si].b;
  t.n0 = blockIdx.y * 128;
  t.kt = min(128, sk1 - t.kg);
  const int kt2 = min(128, a.Ktot - t.kg);   // output rows of the feature outputs C2 (kt = kt2 for gemm_tn's segment tables)
  t.nt = t.sb >= 0 ? max(0, min(128, a.N - t.n0)) : 0;
  t.n2 = (blockIdx.y == 0) ? a.N2 : 0;
  const int ntot = t.nt + t.n2;
  const long long r0 = (long long)blockIdx.z * a.chunk, r1 = min(a.M, r0 + a.chunk);
  const int nchunks = ntot > 0 ? (int)max(0ll, (r1 - r0 + P::ROWS - 1) / P::ROWS) : 0;
  uint8_t* raw = sm;
  uint8_t* cv = sm + TN_NR * P::RAW;
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
    P conv(a, t, tid);
    // running sums of this thread's part of the output tile: row orow, 16-column groups half, half + 2, ...
    const int orow = (warp & 3) * 32 + lane, half = warp >> 2;
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
      release_stage(conv.load(raw + rs * P::RAW), &bar_rfree[rs]);
      if (kc >= TN_NC) mbar_wait(&bar_empty[cs], (uint32_t)((kc / TN_NC - 1) & 1));
      // the MMAs of chunks <= kc - TN_NC have completed: group g is whole once (g + 1) * TN_GROUP - 1 <= kc - TN_NC
      if (kc >= TN_GROUP + TN_NC - 1 && (kc - (TN_NC - 1)) % TN_GROUP == 0) {
        drain(drained & 1);
        ++drained;
      }
      conv.store(cv + cs * P::CV);
      fence_proxy_async();
      mbar_arrive(&bar_full[cs]);
    }
    // ---- epilogue: remaining groups, then the partial tile -> Cp[z] (an empty split contributes zeros) ----
    const int ngroups = (nchunks + TN_GROUP - 1) / TN_GROUP;
    if (nchunks > 0) mbar_wait(&bar_done, 0);
    for (; drained < ngroups; ++drained) drain(drained & 1);
    const bool row_ok = orow < t.kt, row_ok2 = orow < kt2;
    float* cp = t.nt > 0 ? segC + ((size_t)blockIdx.z * (sk1 - sk0) + (t.kg - sk0) + (row_ok ? orow : 0)) * a.N + t.n0 : nullptr;
    float* cp2 = t.n2 ? a.C2 + (size_t)blockIdx.z * a.c2_split + (size_t)(t.kg + (row_ok2 ? orow : 0)) * 32 : nullptr;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int c0 = half * 16 + 32 * i;
      if (c0 < ntot && (c0 < t.nt ? row_ok : row_ok2)) {
        float* o = c0 < t.nt ? cp + c0 : cp2 + (c0 - t.nt);
#pragma unroll
        for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[i][j], acc[i][j + 1], acc[i][j + 2], acc[i][j + 3]);
      }
    }
  } else if (warp == TN_W_MMA) {
    const uint32_t idesc = make_idesc(P::FMT, 128, max(ntot, 16), P::MN, P::MN);
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
        P::mma(tmem + buf * TN_ACC, base + s * P::CV, idesc, kg0 > 0);
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
      if (t.sb >= 0) tmap_prefetch(&a.tb[t.sb]);
      if (t.n2) tmap_prefetch(&a.tf);
      const uint32_t bytes = P::bytes(a, t);
      for (int kc = 0; kc < nchunks; ++kc) {
        const int rs = kc % TN_NR;
        if (kc >= TN_NR) mbar_wait(&bar_rfree[rs], (uint32_t)((kc / TN_NR - 1) & 1));
        mbar_arrive_expect_tx(&bar_raw[rs], bytes);
        P::boxes(raw + rs * P::RAW, a, t, (int)(r0 + (long long)kc * P::ROWS), &bar_raw[rs]);
      }
    }
  }
  __syncthreads();
  if (warp == TN_W_MMA) tmem_dealloc(tmem, 512);
}

__global__ void __launch_bounds__(TN_THREADS, 1) k_gemm_tn_tma(const __grid_constant__ TnArgs a) { gemm_rows<TnTf32>(a); }
__global__ void __launch_bounds__(TN_THREADS, 1) k_gemm_kt(const __grid_constant__ TnArgs a) { gemm_rows<Kt>(a); }
__global__ void __launch_bounds__(TN_THREADS, 1) k_gemm_tn_bf16(const __grid_constant__ TnArgs a) { gemm_rows<TnBf16>(a); }

// fills and checks the segment table: segment s covers columns [seg_k0[s], k1) of A (k1 = seg_k1[s], or the next start and
// Ktot for the last segment when seg_k1 is null) with operand Bs[seg_b[s]] (none when seg_b[s] < 0) and output seg_C[s].
// Segments start at multiples of 128 and follow each other inside [0, Ktot), so a tile's rows past its segment's end
// are past Ktot too.  Returns the operands the segments use (bit b), or -1.
int tn_segments(TnArgs& a, int Ktot, int nseg, const int* seg_k0, const int* seg_k1, const int* seg_b, float* const* seg_C,
                const float* const* Bs, const char* who) {
  int used = 0;
  for (int s = 0; s < nseg; ++s) {
    TnSeg& g = a.seg[s];
    g.k0 = seg_k0[s];
    g.k1 = seg_k1 ? seg_k1[s] : s + 1 < nseg ? seg_k0[s + 1] : Ktot;
    g.b = seg_b[s];
    g.C = seg_C[s];
    REGT_CHECK(g.k0 % 128 == 0 && g.k0 < g.k1 && g.k1 <= Ktot && (s == 0 || g.k0 >= a.seg[s - 1].k1),
               "%s: segment %d [%d, %d) must start at a multiple of 128 after the previous one and end by %d", who, s, g.k0, g.k1, Ktot);
    REGT_CHECK(g.b < 2 && (g.b < 0 || (g.C && Bs[g.b])), "%s: segment %d has no operand / output", who, s);
    if (g.b >= 0) used |= 1 << g.b;
  }
  a.nseg = nseg;
  return used;
}

template <class P>
int launch_rows(void (*kernel)(TnArgs), const char* name, const TnArgs& a, dim3 grid, cudaStream_t st) {
  const size_t smem = (size_t)TN_NR * P::RAW + (size_t)TN_NC * P::CV + 1024;
  REGT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid, TN_THREADS, smem, st>>>(a);
  REGT_LAUNCHED(name, st);
  return 0;
}
}  // namespace

size_t gemm_nt_scratch_floats(int N, int K, GemmKind kind) {
  const int ck = nt_geom(kind).ck;
  const size_t floats = (size_t)((N + 127) / 128 * 128) * ((K + ck - 1) / ck * ck);   // Np x Kp
  return kind == GemmKind::Bf16 ? floats / 2 : 2 * floats;                             // bf16 image, or tf32 hi | lo
}

// C[M][N] = A[M][K] . Bt[N][K]^T for any M >= 1 (TMA zero-fills the rows of the last tile past M; they are not stored);
// `scratch` (gemm_nt_scratch_floats(N, K, kind) floats) receives the hi / lo images of Bt, or its bf16 image.
int launch_gemm_nt_tma(const float* A, long long lda, const float* Bt, long long ldb, float* C, long long ldc, long long M, int N,
                       int K, float* scratch, cudaStream_t st, GemmKind kind) {
  REGT_CHECK(A && Bt && C && scratch && M >= 1 && N > 0 && N % 16 == 0 && K > 0 && K % 4 == 0 && ldc % 4 == 0 &&
                 ((uintptr_t)C % 16) == 0 && ((uintptr_t)scratch % 16) == 0,
             "gemm_nt_tma: bad operands (M=%lld N=%d K=%d)", M, N, K);
  const bool bf16 = kind == GemmKind::Bf16;
  const NtGeom g = nt_geom(kind);
  const int Np = (N + 127) / 128 * 128, Kp = (K + g.ck - 1) / g.ck * g.ck, nchunks = Kp / g.ck;
  NtArgs a{};
  if (bf16) {
    __nv_bfloat16* img = reinterpret_cast<__nv_bfloat16*>(scratch);
    k_pack_bf16<<<cdiv((long long)Np * Kp, 256), 256, 0, st>>>(Bt, ldb, N, K, Np, Kp, img);
    REGT_LAUNCHED("k_pack_bf16", st);
    if (tmap_2d(&a.ta, A, K, M, lda, 128, "gemm_nt_bf16(A)")) return -1;
    if (tmap_2d(&a.tb[0], img, Kp, Np, Kp, 128, "gemm_nt_bf16(B)")) return -1;
  } else {
    float* hi = scratch;
    float* lo = scratch + (size_t)Np * Kp;
    k_split_hilo<<<cdiv((long long)Np * Kp, 256), 256, 0, st>>>(Bt, ldb, N, K, Np, Kp, hi, lo);
    REGT_LAUNCHED("k_split_hilo", st);
    if (tmap_2d(&a.ta, A, K, M, lda, 128, "gemm_nt_tma(A)")) return -1;
    if (tmap_2d(&a.tb[0], hi, Kp, Np, Kp, 128, "gemm_nt_tma(B hi)")) return -1;
    if (tmap_2d(&a.tb[1], lo, Kp, Np, Kp, 128, "gemm_nt_tma(B lo)")) return -1;
  }
  a.C = C; a.M = M; a.ldc = ldc; a.N = N; a.K = K;
  // shared memory: the weights (parked when N <= 128 and they leave room for two stages) + bf16's converted A tiles
  // + the stages of raw fp32 A chunks (and streamed weight tiles)
  a.resident = (N <= 128 && nchunks * g.wt + g.aslots + 2 * 2 * TILE <= SMEM_BUDGET) ? 1 : 0;
  const int fixed = (a.resident ? nchunks * g.wt : 0) + g.aslots;
  const int stage = g.raw_a + (a.resident ? 0 : g.wt);
  a.ns = min(MAXS, (SMEM_BUDGET - fixed) / stage);
  const long long ntiles = (long long)cdiv(M, 128) * cdiv(N, 128);
  const size_t smem = (size_t)fixed + (size_t)a.ns * stage + 1024;
  void (*kernel)(NtArgs) = bf16 ? k_gemm_nt_bf16 : k_gemm_nt_tma_ts;
  REGT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<(int)min(ntiles, (long long)sm_count()), NT_THREADS, smem, st>>>(a);
  REGT_LAUNCHED(bf16 ? "k_gemm_nt_bf16" : "k_gemm_nt_tma_ts", st);
  return 0;
}

// One launch of the row contraction over several column segments of A (each K-tile of 128 columns belongs to one segment):
//   seg s: Cs[z][k1-k0][N] = partials of A[:, k0:k1]^T . B_s      (B_s = Bs[seg_b[s]], or none when seg_b[s] < 0)
//   and, for every segment, C2[z][k0:k1][32] = partials of A[:, k0:k1]^T . B2.
// Segments start at multiples of 128.  kind Bf16: the single-pass bf16 kernel.
int launch_gemm_tn_tma(const float* A, long long lda, long long M, int Ktot, int nseg, const int* seg_k0, const int* seg_b,
                       float* const* seg_C, const float* const* Bs, const long long* ldbs, int N, int splits, const float* B2,
                       long long ldb2, float* C2, long long c2_split, cudaStream_t st, int relu_b, GemmKind kind) {
  REGT_CHECK(A && nseg >= 1 && nseg <= 4 && Ktot % 32 == 0 && N % 32 == 0 && splits > 0 && M >= 1, "gemm_tn_tma: bad shape");
  REGT_CHECK(!B2 || (C2 && ldb2 % 4 == 0), "gemm_tn_tma: bad second operand");
  const bool bf16 = kind == GemmKind::Bf16;
  const int rows = bf16 ? TnBf16::ROWS : TnTf32::ROWS;   // rows per chunk = rows of a TMA box
  TnArgs a{};
  if (tmap_2d(&a.ta, A, Ktot, M, lda, rows, "gemm_tn_tma(A)")) return -1;
  const int used = tn_segments(a, Ktot, nseg, seg_k0, nullptr, seg_b, seg_C, Bs, "gemm_tn_tma");
  if (used < 0) return -1;
  for (int b = 0; b < 2; ++b)
    if ((used >> b & 1) && tmap_2d(&a.tb[b], Bs[b], N, M, ldbs[b], rows, "gemm_tn_tma(B)")) return -1;
  REGT_CHECK(used || B2, "gemm_tn_tma: nothing to contract with");
  if (B2 && tmap_2d(&a.tf, B2, 32, M, ldb2, rows, "gemm_tn_tma(B2)")) return -1;
  a.C2 = C2;
  a.c2_split = c2_split > 0 ? c2_split : (long long)Ktot * 32;
  a.M = M;
  const long long chunk = (M + splits - 1) / splits;
  a.chunk = (chunk + rows - 1) / rows * rows;
  a.Ktot = Ktot;
  a.N = used ? N : 0;
  a.N2 = B2 ? 32 : 0;
  a.relu_b = relu_b;
  const dim3 grid(cdiv(Ktot, 128), max(1, cdiv(a.N, 128)), splits);
  if (bf16) return launch_rows<TnBf16>(k_gemm_tn_bf16, "k_gemm_tn_bf16", a, grid, st);
  return launch_rows<TnTf32>(k_gemm_tn_tma, "k_gemm_tn_tma", a, grid, st);
}

// the row contraction over transposed tiles (k_gemm_kt): AT [ntile][4][Ktot][32], BTs[b] [ntile][4][N][32], FT [ntile][4][32][32];
// segment boundaries are multiples of 128 columns except the end of the last segment with an operand (H = 64: [Dc | dhp])
int launch_gemm_kt(const float* AT, long long ntile, int Ktot, int nseg, const int* seg_k0, const int* seg_k1, const int* seg_b,
                   float* const* seg_C, const float* const* BTs, int N, int splits, const float* FT, float* C2, long long c2_split,
                   cudaStream_t st) {
  REGT_CHECK(AT && nseg >= 1 && nseg <= 4 && Ktot % 128 == 0 && N % 8 == 0 && N >= 16 && N <= 128 && splits > 0 && ntile > 0 && FT && C2,
             "gemm_kt: bad shape (Ktot=%d N=%d)", Ktot, N);
  REGT_CHECK(ntile * 4 * Ktot < (1ll << 31), "gemm_kt: tile count overflows the TMA coordinate");
  TnArgs a{};
  if (tmap_2d(&a.ta, AT, 32, ntile * 4 * Ktot, 32, 128, "gemm_kt(A^T)")) return -1;
  const int used = tn_segments(a, Ktot, nseg, seg_k0, seg_k1, seg_b, seg_C, BTs, "gemm_kt");
  if (used < 0) return -1;
  for (int b = 0; b < 2; ++b)
    if ((used >> b & 1) && tmap_2d(&a.tb[b], BTs[b], 32, ntile * 4 * N, 32, N, "gemm_kt(B^T)")) return -1;
  if (tmap_2d(&a.tf, FT, 32, ntile * 4 * 32, 32, 32, "gemm_kt(F^T)")) return -1;
  a.C2 = C2;
  a.c2_split = c2_split > 0 ? c2_split : (long long)Ktot * 32;
  a.M = ntile * 128;                                 // 128 rows per tile
  a.chunk = (ntile + splits - 1) / splits * 128;     // whole tiles per split
  a.Ktot = Ktot; a.N = N; a.N2 = 32;
  return launch_rows<Kt>(k_gemm_kt, "k_gemm_kt", a, dim3(Ktot / 128, 1, splits), st);
}

// the single-segment form of launch_gemm_tn_tma: Cp[z][K][N] = partials of A[:, :K]^T . B (no B when N == 0)
int launch_gemm_tn(const float* A, long long lda, const float* B, long long ldb, float* Cp, long long M, int K, int N, int splits,
                   cudaStream_t st, const float* B2, long long ldb2, float* Cp2, long long c2_split, int relu_b, GemmKind kind) {
  const int k0 = 0, sb = N > 0 ? 0 : -1;
  float* cs[1] = {Cp};
  const float* bs[2] = {B, nullptr};
  const long long lds[2] = {ldb, 0};
  return launch_gemm_tn_tma(A, lda, M, K, 1, &k0, &sb, cs, bs, lds, N, splits, B2, ldb2, Cp2, c2_split, st, relu_b, kind);
}

// four-segment form used by the cell backward: A = D [M][4H]; segments z|r (B = h), h~ (B = hR), h_pre (B2 only)
static int debug_gemm_tn_multi(const float* A, int64_t lda, int64_t M, int32_t H, const float* B0, const float* B1, float* C0,
                               float* C1, int32_t splits, const float* B2, float* C2, regt_stream_t stream, GemmKind kind) {
  const int k0[3] = {0, 2 * H, 3 * H}, sb[3] = {0, 1, -1};
  float* cs[3] = {C0, C1, nullptr};
  const float* bs[2] = {B0, B1};
  const long long lds[2] = {H, H};
  return launch_gemm_tn_tma(A, lda, M, 4 * H, 3, k0, sb, cs, bs, lds, H, splits, B2, 32, C2, 0, (cudaStream_t)stream, 0, kind);
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
// the single-pass bf16 forms of the two hooks above (tests/test_gpu_bf16_widths.py); scratch: gemm_nt_scratch_floats(N, K, Bf16)
// floats, which the tf32 hook's scratch size covers
extern "C" int regt_debug_gemm_nt_bf16(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc, int64_t M,
                                       int32_t N, int32_t K, float* scratch, regt_stream_t stream) {
  return regt::launch_gemm_nt_tma(A, lda, Bt, ldb, C, ldc, M, N, K, scratch, (cudaStream_t)stream, regt::GemmKind::Bf16);
}
extern "C" int regt_debug_gemm_tn_bf16(const float* A, int64_t lda, const float* B, int64_t ldb, float* Cp, int64_t M, int32_t K,
                                       int32_t N, int32_t splits, const float* B2, int64_t ldb2, float* Cp2, regt_stream_t stream) {
  return regt::launch_gemm_tn(A, lda, B, ldb, Cp, M, K, N, splits, (cudaStream_t)stream, B2, ldb2, Cp2, 0, 0, regt::GemmKind::Bf16);
}
extern "C" int regt_debug_gemm_tn_multi(const float* A, int64_t lda, int64_t M, int32_t H, const float* B0, const float* B1,
                                        float* C0, float* C1, int32_t splits, const float* B2, float* C2, regt_stream_t stream) {
  return regt::debug_gemm_tn_multi(A, lda, M, H, B0, B1, C0, C1, splits, B2, C2, stream, regt::GemmKind::Tf32x3);
}
extern "C" int regt_debug_gemm_tn_multi_bf16(const float* A, int64_t lda, int64_t M, int32_t H, const float* B0, const float* B1,
                                             float* C0, float* C1, int32_t splits, const float* B2, float* C2, regt_stream_t stream) {
  return regt::debug_gemm_tn_multi(A, lda, M, H, B0, B1, C0, C1, splits, B2, C2, stream, regt::GemmKind::Bf16);
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
