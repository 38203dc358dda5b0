// gemm.cu -- the Linear layers of the denoiser (90 nn.Linear calls per forward in the reference,
// sequence_model/model.py:200-237 via HF BertAttention/BertLayer + SELayer + AminoAcidPredictor).
//
//   C[M,N] = epilogue( A[M,K] * W[N,K]^T + bias[N] (+ resid[M,N]) )
//
// nn.Linear keeps W as [out,in] = [N,K] row-major, i.e. K-major for the MMA B operand; activations are
// [tokens, features] = K-major for the A operand.  No transposes anywhere.
//
// bf16 path (the product): persistent, warp-specialised tcgen05 kernel
//   warp 0      TMA producer   : cp.async.bulk.tensor 2D tiles (128B swizzle) into a STAGES-deep smem ring
//   warp 1      MMA issuer     : one elected thread issues tcgen05.mma (128 x BN x 16, bf16 -> f32 in TMEM);
//                                owns the TMEM allocation (2 accumulator stages = 2*BN columns)
//   warps 2..9  epilogue       : tcgen05.ld the finished accumulator (lane quarter = warp%4, column half =
//                                (warp-2)/4), fused bias / erf-GELU / SiLU / fp32 residual add, 16-bit or fp32
//                                stores -- overlapped with the MMA mainloop of the next tile (double-buffered TMEM).
// Operands are 16-bit (bf16 or fp16, selected through the instruction descriptor; both operands of one MMA
// must share the format); GEMMs that feed a LayerNorm write fp32 and take an fp32 residual, so the residual stream of the
// network never passes through a 16-bit rounding.
// fp32 path (parity gate 1e-5): plain SIMT tiled kernel, fp32 FMA accumulation.
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <type_traits>
#include <unordered_map>

#include "common.cuh"
#include "kernels.h"

namespace seqdiff {

// =====================================================================================================
// TMA descriptors (host)
// =====================================================================================================
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

struct TmapKey {
  const void* ptr;
  int rows, cols, box_rows, fmt;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && box_rows == o.box_rows && fmt == o.fmt;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h ^= (static_cast<size_t>(k.rows) * 0x9E3779B97F4A7C15ull) ^ (static_cast<size_t>(k.cols) << 20) ^ (static_cast<size_t>(k.box_rows) << 44) ^
         (static_cast<size_t>(k.fmt) << 60);
    return h;
  }
};

// row-major 16-bit matrix [rows, cols] (fmt 0 = fp16, 1 = bf16); tile = box_rows x 64 columns, 128B-swizzled,
// OOB reads give zeros
int make_tmap(const void* ptr, int fmt, int rows, int cols, int box_rows, CUtensorMap* out) {
  static std::mutex mu;
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  TmapKey key{ptr, rows, cols, box_rows, fmt};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return SEQDIFF_OK;
    }
  }
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return SEQDIFF_ERR_CUDA;
  }
  SD_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (cols % 8) == 0, "TMA operand must be 16B aligned with a 16B-multiple row pitch");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(cols) * 2};
  cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(out, fmt == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim,
                   gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
    return SEQDIFF_ERR_CUDA;
  }
  std::lock_guard<std::mutex> g(mu);
  cache.emplace(key, *out);
  return SEQDIFF_OK;
}

// Output tile map of the 16-bit GEMM epilogue: row-major [rows, cols], boxes of 32 rows x 32 columns (64 B rows, SWIZZLE_64B).
// Rows past `rows` are clipped by the TMA store, so the epilogue needs no bounds checks.  Cached like make_tmap.
int make_tmap_store16(const void* ptr, int fmt, int rows, int cols, CUtensorMap* out) {
  static std::mutex mu;
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  TmapKey key{ptr, rows, cols, -32, fmt};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return SEQDIFF_OK;
    }
  }
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return SEQDIFF_ERR_CUDA;
  }
  SD_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (cols % 32) == 0, "TMA store operand must be 16B aligned with N a multiple of 32");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(cols) * 2};
  cuuint32_t box[2] = {32u, 32u};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(out, fmt == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim,
                   gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (store) failed with CUresult " + std::to_string(static_cast<int>(r)));
    return SEQDIFF_ERR_CUDA;
  }
  std::lock_guard<std::mutex> g(mu);
  cache.emplace(key, *out);
  return SEQDIFF_OK;
}

// [B][rows][cols] 16-bit tensor (cols contiguous): boxes of 1 x box_rows x 64 columns, 128B swizzle.  Used for TMA STORES of
// per-graph tiles: rows past `rows` are clipped per graph instead of spilling into the next graph's rows.
int make_tmap_3d(const void* ptr, int fmt, int batch, int rows, int cols, int box_rows, CUtensorMap* out) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return SEQDIFF_ERR_CUDA;
  }
  SD_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (cols % 8) == 0, "TMA operand must be 16B aligned with a 16B-multiple row pitch");
  cuuint64_t gdim[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(batch)};
  cuuint64_t gstride[2] = {static_cast<cuuint64_t>(cols) * 2, static_cast<cuuint64_t>(rows) * cols * 2};
  cuuint32_t box[3] = {64u, static_cast<cuuint32_t>(box_rows), 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = enc(out, fmt == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), gdim,
                   gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (3d) failed with CUresult " + std::to_string(static_cast<int>(r)));
    return SEQDIFF_ERR_CUDA;
  }
  return SEQDIFF_OK;
}

// =====================================================================================================
// tcgen05 kernel
// =====================================================================================================
constexpr int kBM = 128;        // UMMA M (one TMEM lane per output row)
constexpr int kBK = 64;         // 64 bf16 = 128 B = one swizzle row
constexpr int kUmmaK = 16;      // K per tcgen05.mma for 16-bit inputs
constexpr int kGemmThreads = 320;

// CG2 = CTA pair (cluster of 2, tcgen05 cta_group::2): one 256 x BN output tile per pair; each CTA stages its own 128 rows
// of A and HALF of the B tile (the MMA reads both halves across the pair), so a CTA pulls 16 KB + BN/2 * 128 B per k-block
// from L2 for 128 x BN x 64 MACs -- 2/3 of the 1-CTA traffic at BN = 256.  The mainloop of this model's GEMMs is bound by
// exactly that L2 -> SM operand stream (profiles/prof_gemm_r01.summary.txt).
template <int BN, bool CG2> struct GemmCfg {
  static_assert(BN <= 256, "one tcgen05.mma per k-step: N <= 256");
  static constexpr int kBoxRows = CG2 ? BN / 2 : BN;  // B rows staged per CTA per k-block (one TMA box)
  static constexpr int kABytes = kBM * kBK * 2;
  static constexpr int kBBytes = kBoxRows * kBK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (CG2 || BN == 128) ? 6 : 4;
  static constexpr int kTmemCols = BN == 128 ? 256 : 512;  // 2 accumulator stages, rounded up to a power of two
  static constexpr int kStagingBytes = 8 * 32 * 32 * 4;  // one 32x32 fp32 transpose panel per epilogue warp
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/ + kStagingBytes;
  static_assert(kSmemBytes <= 232448, "over the 227 KB shared-memory limit");
};

template <typename T> __device__ __forceinline__ void store4(T* p, const float4& v);
template <> __device__ __forceinline__ void store4<float>(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
template <> __device__ __forceinline__ void store4<bf16>(bf16* p, const float4& v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
}
template <> __device__ __forceinline__ void store4<f16>(f16* p, const float4& v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_f16x2(v.x, v.y), pack_f16x2(v.z, v.w));
}

// Epilogue operand loads (the bias of the 16-bit epilogue, the fp32 residual): coherent loads, deliberately not ld.global.nc.  They
// cannot move above the fences and barrier waits around them, so each chunk's registers stay local to its chunk.  With non-coherent
// loads the scheduler hoists them across the unrolled chunk loop: the 16-bit epilogue grows from 86 to 168 registers and spills at
// BN = 256, and the residual epilogue spills more at its 168-register cap.
__device__ __forceinline__ float4 ld_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// split-K partial products: one 128-bit vector atomic per 4 outputs (fp32 C only; the other instantiations never reach it)
template <typename T> __device__ __forceinline__ void add4(T*, const float4&) {}
template <> __device__ __forceinline__ void add4<float>(float* p, const float4& v) { atomicAdd(reinterpret_cast<float4*>(p), v); }

// TOut: bf16 / f16 (operand for the next GEMM or attention) or float (LayerNorm input); resid is always fp32.
// RESID: 0 none, 1 fp32 residual tensor, 2 residual = LayerNorm(resid) rebuilt from per-row (mean, rstd) + affine (g, b)
// TN: C[M,N] = At^T Bt with At [K, M] and Bt [K, N] row-major (both operands MN-major for the MMA): the weight-gradient product
// dW = dY^T X straight from the row-major activations / gradients -- no transposed copies.  tmA / tmB then carry boxes of
// 64 k-rows x 64 columns; K (the token count) may be ragged, rows past it are zero-filled by TMA.
template <int BN, int EPI, int RESID, typename TOut, bool CG2, bool TN = false>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                    const float* __restrict__ bias, const float* __restrict__ resid, TOut* __restrict__ C, int M, int N, int K,
                    uint32_t idesc, const float2* __restrict__ ln_stats, const float* __restrict__ ln_g, const float* __restrict__ ln_b,
                    unsigned long long* __restrict__ trace, int ksplit) {
  // ksplit > 1 (fp32 C without residual only): split-K.  A scheduled tile is (output tile, k-range); every split ADDS its partial
  // product into C with vector atomics (C pre-zeroed by the caller, bias added by split 0).  For the weight-gradient products
  // dW[N,K] = dY^T X of the training step, whose outputs are a few dozen tiles with a contraction over every token of the batch.
  using Cfg = GemmCfg<BN, CG2>;
  static_assert(!TN || (!CG2 && RESID == 0 && EPI == 0 && std::is_same<TOut, float>::value && BN % 64 == 0), "TN: 1-CTA MMA, fp32 C");
  constexpr int STAGES = Cfg::kStages;
  constexpr int TILE_M = CG2 ? 2 * kBM : kBM;  // rows per scheduled tile (per CTA pair / per CTA)
  extern __shared__ uint8_t smem_raw[];
  // 1024B-align by OFFSET (not through an integer cast): keeps the pointer provably shared, so accesses compile to LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tfull_bar = bars + 2 * STAGES;
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = warp_id_uniform();  // provably warp-uniform: the TMA / MMA role loops below stay on the uniform datapath
  const int lane = threadIdx.x & 31;
  const int num_n = N / BN;
  const int num_m = (M + TILE_M - 1) / TILE_M;
  const int num_tiles = num_m * num_n * ksplit;
  const int num_kb = (K + kBK - 1) / kBK;
  auto kb_lo = [&](int ks) { return static_cast<int>(static_cast<long long>(num_kb) * ks / ksplit); };
  const uint32_t cta_rank = CG2 ? cluster_ctarank() : 0u;  // 0 = leader (issues the MMAs), 1 = peer
  const int tile0 = CG2 ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = CG2 ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);

  // optional timeline (debug, seqdiff_debug_attn_trace): CTA 0, lane 0 of the TMA / MMA / two epilogue warps
  int tr_n = 0;
  const bool tr_on = trace != nullptr && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 1 || warp == 2 || warp == 6);
  const int tr_base = (warp == 0 ? 0 : warp == 1 ? 1 : warp == 2 ? 2 : 3) * 1024;
  auto TR = [&](int id) {
    if (tr_on && tr_n < 1023) trace[tr_base + 1 + tr_n++] = (static_cast<unsigned long long>(clock64()) << 8) | static_cast<unsigned>(id);
  };
  TR(40);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (!std::is_same<TOut, float>::value) tma_prefetch_desc(&tmC);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], CG2 ? 16 : 8);  // one arrival per epilogue warp (of both CTAs of a pair)
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (CG2) {
      tmem_alloc_cg2(tmem_slot, Cfg::kTmemCols);  // collective over the pair: same warp, same slot in both CTAs
      tmem_relinquish_cg2();
    } else {
      tmem_alloc(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (CG2) cluster_sync_all(); else __syncthreads();  // barriers of both CTAs of a pair initialised before any remote arrive / TMA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  TR(41);
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  TR(42);

  if (warp == 0) {
    // ------------------------------- TMA producer -------------------------------
    // (whole warp runs the loop; one elected lane issues -- see common.cuh "warp-uniform single-issuer variants")
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        const int ks = tile % ksplit, mn = tile / ksplit;
        const int m_blk = mn / num_n, n_blk = mn % num_n;
        const int a_row = m_blk * TILE_M + static_cast<int>(cta_rank) * kBM;
        for (int kb = kb_lo(ks), kb_end = kb_lo(ks + 1); kb < kb_end; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          TR(1);
          if (CG2) {
            // both CTAs' tiles complete on the LEADER's full barrier, which the leader arms for the bytes of the pair
            if (cta_rank == 0) mbar_expect_tx_e(&full_bar[stage], 2 * Cfg::kStageBytes);
            const uint32_t bar = mapa_u32(smem_u32(&full_bar[stage]), 0);
            tma_load_2d_cg2_e(sA + stage * Cfg::kABytes, &tmA, bar, kb * kBK, a_row);
            // half of the UMMA's B tile lives in each CTA of the pair
            tma_load_2d_cg2_e(sB + stage * Cfg::kBBytes, &tmB, bar, kb * kBK, n_blk * BN + static_cast<int>(cta_rank) * Cfg::kBoxRows);
          } else if (TN) {
            mbar_expect_tx_e(&full_bar[stage], Cfg::kStageBytes);
#pragma unroll
            for (int j = 0; j < kBM / 64; ++j)  // A^T: 64-column blocks of the M (= output row) range, 64 k-rows each
              tma_load_2d_e(sA + stage * Cfg::kABytes + j * 8192, &tmA, &full_bar[stage], a_row + 64 * j, kb * kBK);
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_2d_e(sB + stage * Cfg::kBBytes + j * 8192, &tmB, &full_bar[stage], n_blk * BN + 64 * j, kb * kBK);
          } else {
            mbar_expect_tx_e(&full_bar[stage], Cfg::kStageBytes);
            tma_load_2d_e(sA + stage * Cfg::kABytes, &tmA, &full_bar[stage], kb * kBK, a_row);
            tma_load_2d_e(sB + stage * Cfg::kBBytes, &tmB, &full_bar[stage], kb * kBK, n_blk * BN);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer ---------------------------------
    if (cta_rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        mbar_wait(&tempty_bar[as], aphase ^ 1);  // epilogue(s) have drained this accumulator stage
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(as * BN);
        const int kb_begin = kb_lo(tile % ksplit), kb_end = kb_lo(tile % ksplit + 1);
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          TR(11);
          const uint32_t a_addr = smem_u32(sA + stage * Cfg::kABytes);
          const uint32_t b_addr = smem_u32(sB + stage * Cfg::kBBytes);
#pragma unroll
          for (int k = 0; k < kBK / kUmmaK; ++k) {
            const uint64_t adesc = TN ? umma_desc_mnmajor_sw128(a_addr + k * 2048, 8192) : umma_desc_kmajor_sw128(a_addr + k * kUmmaK * 2);
            const uint64_t bdesc = TN ? umma_desc_mnmajor_sw128(b_addr + k * 2048, 8192) : umma_desc_kmajor_sw128(b_addr + k * kUmmaK * 2);
            if (CG2) umma_cg2_e(tmem_d, adesc, bdesc, idesc, ((kb - kb_begin) | k) != 0 ? 1u : 0u);
            else umma_bf16_e(tmem_d, adesc, bdesc, idesc, ((kb - kb_begin) | k) != 0 ? 1u : 0u);
          }
          // smem slot reusable once these MMAs have read it (in both CTAs of a pair)
          if (CG2) umma_commit_mc_e(&empty_bar[stage], 3); else umma_commit_e(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (CG2) umma_commit_mc_e(&tfull_bar[as], 3); else umma_commit_e(&tfull_bar[as]);  // accumulator complete -> epilogue(s)
        TR(12);
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else {
    // ------------------------------- epilogue -----------------------------------
    // Accumulators arrive one TMEM lane (= output row) per thread.  Each 32x32 chunk is transposed through a
    // per-warp smem panel (128 B rows, 16 B chunks XOR-swizzled by row&7: conflict-free both ways) so that
    // bias / activation / residual / store run with 8 lanes per row segment: every global instruction touches
    // 4 cache lines instead of 32, bias is one float4 per chunk, and the fp32 residual is prefetched before the
    // TMEM load is waited on.
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;  // column half of the tile
    float* stage = reinterpret_cast<float*>(smem + STAGES * Cfg::kStageBytes + 256) + (warp - 2) * 1024;
    const int lr = lane >> 3, lc = lane & 7;
    int as = 0;
    uint32_t aphase = 0;
    constexpr bool kTmaOut = !std::is_same<TOut, float>::value && RESID == 0;  // 16-bit output tiles leave through TMA stores
    int pcount = 0;  // staging panels used so far (they alternate across chunks AND tiles)
    (void)pcount;
    constexpr int NCH = BN / 64;  // 32-column chunks per warp and tile
    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
      const int ks = tile % ksplit, mn = tile / ksplit;
      const int m_blk = mn / num_n, n_blk = mn % num_n;
      const int row_base = m_blk * TILE_M + static_cast<int>(cta_rank) * kBM + q * 32;
      SD_DEV_ASSERT(m_blk < num_m && n_blk * BN + half * (BN / 2) + (BN / 2) <= N && ks < ksplit);  // the tile decode stays inside C
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * BN) + half * (BN / 2);
      const int col0 = n_blk * BN + half * (BN / 2) + 4 * lc;  // this lane's 4 columns of chunk 0; chunk ci adds 32 ci
      const bool full = row_base + 32 <= M;                    // warp-uniform: no row of this warp's slab is out of range
      if constexpr (kTmaOut) {
        // ---- 16-bit outputs without residual: no transpose.  Each thread owns one accumulator row (TMEM lane) and 32
        // columns per chunk: bias (broadcast loads) / activation / pack, 64 B per row into a SWIZZLE_64B panel, one TMA
        // store per 32 x 32 chunk.  Per-lane STG of the transposed layout went through the LSU / L1TEX path shared with the
        // operand fills and slowed the concurrent mainloop by 20 % (timelines with the stores removed: 8.1 k -> 6.75 k cycles
        // per 128 x 256 x 768 tile); the bulk store leaves the SM through the async proxy, rows past M are clipped by the map.
        const int colw = n_blk * BN + half * (BN / 2);  // first column of this warp's slab
        uint8_t* panels = reinterpret_cast<uint8_t*>(stage);  // this warp's 4 KB: two 32 x 64 B panels
        TR(20);
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        TR(21);
        uint32_t r[2][32];
        tmem_ld_32x32(t_row, r[0]);
#pragma unroll
        for (int ci = 0; ci < NCH; ++ci) {
          const int cur = ci & 1;
          float4 bv[8];
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) bv[j4] = ld_f4(bias + colw + 32 * ci + 4 * j4);  // same address in every lane
          tmem_ld_wait();
          if (ci + 1 < NCH) tmem_ld_32x32(t_row + static_cast<uint32_t>(32 * (ci + 1)), r[cur ^ 1]);
          uint32_t pk[16];
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            float a0 = __uint_as_float(r[cur][4 * j4]) + bv[j4].x, a1 = __uint_as_float(r[cur][4 * j4 + 1]) + bv[j4].y;
            float a2 = __uint_as_float(r[cur][4 * j4 + 2]) + bv[j4].z, a3 = __uint_as_float(r[cur][4 * j4 + 3]) + bv[j4].w;
            if (EPI == 1) { a0 = gelu_fast(a0); a1 = gelu_fast(a1); a2 = gelu_fast(a2); a3 = gelu_fast(a3); }
            if (EPI == 2) { a0 = silu_fast(a0); a1 = silu_fast(a1); a2 = silu_fast(a2); a3 = silu_fast(a3); }
            pk[2 * j4] = pack2<TOut>(a0, a1);
            pk[2 * j4 + 1] = pack2<TOut>(a2, a3);
          }
          uint8_t* panel = panels + (pcount & 1) * 2048;
          if (lane == 0) tma_store_wait_read1();  // the store that last used this panel (two chunks ago) has read it
          __syncwarp();
          // SWIZZLE_64B: 16 B chunk index XOR bits [7:8] of the ABSOLUTE shared address (the panels sit 256 B past a 1 KB
          // boundary, behind the barrier block, so the pattern is not simply a function of the row number)
          uint8_t* prow = panel + lane * 64;
          const uint32_t sw = (smem_u32(prow) >> 7) & 3u;
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16)
            *reinterpret_cast<uint4*>(prow + ((static_cast<uint32_t>(c16) ^ sw) << 4)) =
                make_uint4(pk[4 * c16], pk[4 * c16 + 1], pk[4 * c16 + 2], pk[4 * c16 + 3]);
          fence_proxy_async_smem();  // generic-proxy writes -> visible to the TMA store (async proxy)
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmC, panel, colw + 32 * ci, row_base);
            tma_store_commit();
          }
          ++pcount;
        }
      } else {
      // Everything the tile needs from global memory that does not depend on the accumulator is fetched BEFORE the wait
      // on the MMAs (LayerNorm row statistics, the first chunk's bias / residual); inside the chunk loop the next chunk's
      // bias / residual / LayerNorm affine and the next chunk's TMEM load are in flight while the current chunk is transposed and
      // stored.  (Timeline before: 1450 cycles per chunk, i.e. an epilogue as long as a K = 768 mainloop.)
      float2 st8[8];
      if (RESID == 2) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int row = row_base + 4 * i + lr;
          st8[i] = row < M ? __ldg(ln_stats + row) : make_float2(0.f, 0.f);
        }
      }
      // bias / LayerNorm affine of a chunk: double-buffered, fetched one chunk ahead.  Residual: ONE buffer of 8 float4, each
      // entry re-filled for the next chunk right after it has been consumed (a second buffer costs 32 registers and spills).
      float4 rres[8], g4[2], h4[2], b4[2];
      auto fetch_small = [&](int ci, int buf) {
        b4[buf] = ks == 0 ? __ldg(reinterpret_cast<const float4*>(bias + col0 + 32 * ci)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (RESID == 2) {
          g4[buf] = __ldg(reinterpret_cast<const float4*>(ln_g + col0 + 32 * ci));
          h4[buf] = __ldg(reinterpret_cast<const float4*>(ln_b + col0 + 32 * ci));
        }
      };
      auto fetch_resid_row = [&](int ci, int i) {
        const int row = row_base + 4 * i + lr;
        rres[i] = (full || row < M) ? ld_f4(resid + static_cast<size_t>(row) * N + col0 + 32 * ci)
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      fetch_small(0, 0);
      if (RESID) {
#pragma unroll
        for (int i = 0; i < 8; ++i) fetch_resid_row(0, i);
      }
      TR(20);
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      TR(21);
      // the TMEM load is double-buffered only without a residual (the residual prefetch already takes 32 registers per
      // buffer and the kernel is capped at 168: 320 threads are allocated as 12 warps)
      constexpr bool kPrefT = RESID == 0;
      uint32_t r[kPrefT ? 2 : 1][32];
      if (kPrefT) tmem_ld_32x32(t_row, r[0]);
#pragma unroll
      for (int ci = 0; ci < NCH; ++ci) {
        const int cur = ci & 1;
        const int tc = kPrefT ? cur : 0;
        if (ci + 1 < NCH) fetch_small(ci + 1, cur ^ 1);
        if (!kPrefT) tmem_ld_32x32(t_row + static_cast<uint32_t>(32 * ci), r[0]);
        tmem_ld_wait();
        if (kPrefT && ci + 1 < NCH) tmem_ld_32x32(t_row + static_cast<uint32_t>(32 * (ci + 1)), r[tc ^ 1]);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj)
          *reinterpret_cast<uint4*>(stage + lane * 32 + ((jj ^ (lane & 7)) << 2)) =
              make_uint4(r[tc][4 * jj], r[tc][4 * jj + 1], r[tc][4 * jj + 2], r[tc][4 * jj + 3]);
        __syncwarp();
        const int col = col0 + 32 * ci;
        // rows in two groups of four: the four smem reads of a group are issued back to back (one dependent chain per row
        // serialised the whole chunk on LDS latency) and the stores of a full tile carry no per-row bounds branch
        auto emit_rows = [&](auto guard_tag) {
          constexpr bool kGuard = decltype(guard_tag)::value;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int rr = 4 * (4 * hh + u) + lr;
              v[u] = *reinterpret_cast<const float4*>(stage + rr * 32 + ((lc ^ (rr & 7)) << 2));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int i = 4 * hh + u;
              v[u].x += b4[cur].x; v[u].y += b4[cur].y; v[u].z += b4[cur].z; v[u].w += b4[cur].w;
              if (EPI == 1) { v[u].x = gelu_fast(v[u].x); v[u].y = gelu_fast(v[u].y); v[u].z = gelu_fast(v[u].z); v[u].w = gelu_fast(v[u].w); }
              if (EPI == 2) { v[u].x = silu_fast(v[u].x); v[u].y = silu_fast(v[u].y); v[u].z = silu_fast(v[u].z); v[u].w = silu_fast(v[u].w); }
              if (RESID) {
                float4 rv = rres[i];
                if (ci + 1 < NCH) fetch_resid_row(ci + 1, i);  // refill this slot for the next chunk
                if (RESID == 2) {  // residual = LayerNorm(resid row): same fp32 formula and op order as layernorm_kernel
                  rv.x = (rv.x - st8[i].x) * st8[i].y * g4[cur].x + h4[cur].x;
                  rv.y = (rv.y - st8[i].x) * st8[i].y * g4[cur].y + h4[cur].y;
                  rv.z = (rv.z - st8[i].x) * st8[i].y * g4[cur].z + h4[cur].z;
                  rv.w = (rv.w - st8[i].x) * st8[i].y * g4[cur].w + h4[cur].w;
                }
                v[u].x += rv.x; v[u].y += rv.y; v[u].z += rv.z; v[u].w += rv.w;
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int row = row_base + 4 * (4 * hh + u) + lr;
              if (!kGuard || row < M) {
                if (std::is_same<TOut, float>::value && RESID == 0 && ksplit > 1) add4(C + static_cast<size_t>(row) * N + col, v[u]);
                else store4<TOut>(C + static_cast<size_t>(row) * N + col, v[u]);
              }
            }
          }
        };
        if (full) emit_rows(std::false_type{}); else emit_rows(std::true_type{});
        __syncwarp();
      }
      }
      TR(23);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG2 && cta_rank != 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[as]), 0));  // the leader's MMA thread waits on it
        else mbar_arrive(&tempty_bar[as]);
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (kTmaOut && lane == 0) tma_store_wait_all();  // bulk stores complete (and visible) before the CTA exits
  }

  TR(43);
  if (tr_on) trace[tr_base] = static_cast<unsigned long long>(tr_n);
  tc_fence_before();
  if (CG2) cluster_sync_all(); else __syncthreads();  // pair: nobody frees TMEM / exits while the peer may still signal, read or write here
  if (warp == 1) {
    tc_fence_after();
    if (CG2) tmem_dealloc_cg2(tmem_base, Cfg::kTmemCols); else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, int EPI, int RESID, typename TOut, bool CG2>
static int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const float* bias, const float* resid, void* C, int M,
                     int N, int K, uint32_t idesc, cudaStream_t s, const LnResid* ln = nullptr, int ksplit = 1) {
  using Cfg = GemmCfg<BN, CG2>;
  auto kfn = gemm_tcgen05_kernel<BN, EPI, RESID, TOut, CG2>;
  static bool configured = false;  // per instantiation
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  const int tiles = ceil_div(M, CG2 ? 2 * kBM : kBM) * (N / BN) * ksplit;
  const int slots = CG2 ? num_sms() / 2 : num_sms();
  const int grid = (tiles < slots ? tiles : slots) * (CG2 ? 2 : 1);
  SD_CUDA(launch_kc(CG2 ? 2 : 1, kfn, dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, s, ta, tb, tc, bias, resid, static_cast<TOut*>(C), M, N, K,
                    idesc, ln ? ln->stats : nullptr, ln ? ln->g : nullptr, ln ? ln->b : nullptr, g_attn_trace, ksplit));
  SD_LAUNCHED(ksplit > 1 ? (CG2 ? "gemm_tcgen05_2cta_splitk" : "gemm_tcgen05_splitk") : (CG2 ? "gemm_tcgen05_2cta" : "gemm_tcgen05"), s);
  return SEQDIFF_OK;
}

// C[M,N] (+)= At^T Bt: At [K, M], Bt [K, N] row-major 16-bit (fmt 0 = fp16, 1 = bf16), fp32 C.  split_k as in gemm_16 (C pre-zeroed when != 1).
template <int BN>
static int launch_tn(const CUtensorMap& ta, const CUtensorMap& tb, const float* bias, float* C, int M, int N, int K, uint32_t idesc, int ksplit, cudaStream_t s) {
  using Cfg = GemmCfg<BN, false>;
  auto kfn = gemm_tcgen05_kernel<BN, 0, 0, float, false, true>;
  static bool configured = false;
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  const int tiles = ceil_div(M, kBM) * (N / BN) * ksplit;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  SD_CUDA(launch_kc(1, kfn, dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, s, ta, tb, ta, bias, static_cast<const float*>(nullptr), C, M, N, K, idesc,
                    static_cast<const float2*>(nullptr), static_cast<const float*>(nullptr), static_cast<const float*>(nullptr), g_attn_trace, ksplit));
  SD_LAUNCHED(ksplit > 1 ? "gemm_tcgen05_tn_splitk" : "gemm_tcgen05_tn", s);
  return SEQDIFF_OK;
}
int gemm_16_tn(int M, int N, int K, const void* At, const void* Bt, int fmt, const float* bias, float* C, cudaStream_t s, int split_k) {
  SD_CHECK(M > 0 && N > 0 && K > 0, "empty GEMM");
  SD_CHECK(M % 8 == 0 && N % 128 == 0, "TN GEMM: M % 8 == 0 (16B TMA pitch) and N % 128 == 0");
  SD_CHECK((fmt | 1) == 1 && bias != nullptr, "bad operand format / bias required");
  SD_CHECK(split_k >= -1 && split_k != 0, "split_k must be -1 (auto), 1 (off) or the number of k-ranges");
  const int bn = N % 256 == 0 ? 256 : 128;
  int ksplit = split_k;
  const int nkb = ceil_div(K, kBK);
  if (ksplit < 0) {
    const int tiles = ceil_div(M, kBM) * (N / bn);
    ksplit = num_sms() / tiles;
    if (ksplit > nkb / 4) ksplit = nkb / 4;
  }
  if (ksplit > nkb) ksplit = nkb;
  if (ksplit < 1) ksplit = 1;
  CUtensorMap ta, tb;
  SD_TRY(make_tmap(At, fmt, K, M, 64, &ta));  // boxes of 64 k-rows x 64 columns
  SD_TRY(make_tmap(Bt, fmt, K, N, 64, &tb));
  const uint32_t idesc = umma_idesc_16(kBM, bn, static_cast<uint32_t>(fmt), static_cast<uint32_t>(fmt)) | kUmmaAMnMajor | kUmmaBMnMajor;
  if (bn == 256) return launch_tn<256>(ta, tb, bias, C, M, N, K, idesc, ksplit, s);
  return launch_tn<128>(ta, tb, bias, C, M, N, K, idesc, ksplit, s);
}

// tile choice, from measurements on B200 (scripts/gemm_sweep.py, profiles/gemm_sweep_r01.log):
//  * the mainloop is bound by the L2->SM operand stream, so wide tiles win: 128x256 (48 KB of operands per 128x256x64 MACs)
//    beats 128x128 (32 KB per half the MACs) on every shape of this model;
//  * 128x192 exists for wave quantisation: N = 768 at M = 8192 is 192 tiles of 128x256 (2 waves at 65 % fill on 148 SMs) but
//    256 tiles of 128x192 (2 waves of 3/4-size tiles);
//  * CTA pairs (cta_group::2, 256x256 per pair, 32 KB per CTA for the same MACs) gain 5-7 % on the largest GEMMs
//    (ada2 1.21, cross-KV 1.23 PFLOP/s) and nothing on the small ones, whose time is ramp / tail: used from 2.5e10 MACs up.
// Returns bn | (cg2 << 16).
static int pick_cfg(int M, int N, int K) {
  if (M <= 64) return 128;
  if (N % 256 == 0 && static_cast<double>(M) * N * K >= 2.5e10) return 256 | (1 << 16);
  const int sms = num_sms();
  const int m_tiles = ceil_div(M, kBM);
  int best = 0;
  double best_cost = 0;
  for (int bn : {256, 192, 128}) {
    if (N % bn) continue;
    const int waves = ceil_div(m_tiles * (N / bn), sms);
    const double cost = waves * bn * (1.0 + 48.0 / bn);  // per-tile time ~ bn, with a bandwidth penalty for narrow tiles
    if (!best || cost < best_cost * 0.97) { best = bn; best_cost = cost; }
  }
  return best;
}

template <int BN, bool CG2>
static int dispatch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const float* bias, const float* resid, int epi, void* C,
                       int out_kind, int M, int N, int K, uint32_t idesc, cudaStream_t s, const LnResid* ln, int ksplit = 1) {
  if (resid && ln) return launch_tc<BN, 0, 2, float, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s, ln);
  if (resid) return launch_tc<BN, 0, 1, float, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
  if (out_kind == 2) return launch_tc<BN, 0, 0, float, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s, nullptr, ksplit);
  if (out_kind == 1) {
    if (epi == 0) return launch_tc<BN, 0, 0, bf16, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
    if (epi == 1) return launch_tc<BN, 1, 0, bf16, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
    return launch_tc<BN, 2, 0, bf16, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
  }
  if (epi == 0) return launch_tc<BN, 0, 0, f16, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
  if (epi == 1) return launch_tc<BN, 1, 0, f16, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
  return launch_tc<BN, 2, 0, f16, CG2>(ta, tb, tc, bias, resid, C, M, N, K, idesc, s);
}

// a_fmt / w_fmt: 0 = fp16, 1 = bf16.  out_kind: 0 = fp16, 1 = bf16, 2 = fp32 (identity epilogue only; implied by resid).
// force_cfg: 0 = auto, else  bn | (cg2 << 16)  with bn in {128,192,256} (tests / sweeps).
int gemm_16(int M, int N, int K, const void* A, int a_fmt, const void* W, int w_fmt, const float* bias, const float* resid, int epi,
            void* C, int out_kind, cudaStream_t s, int force_cfg, const LnResid* ln_resid, int split_k) {
  SD_CHECK(M > 0 && N > 0 && K > 0, "empty GEMM");
  // split_k: 1 = off; n > 1 = n k-ranges per output tile; -1 = as many as fill the GPU (>= 4 k-blocks each).  C must be pre-zeroed.
  SD_CHECK(split_k >= -1 && split_k != 0, "split_k must be -1 (auto), 1 (off) or the number of k-ranges");
  SD_CHECK(split_k == 1 || (out_kind == 2 && !resid && epi == 0), "split-K accumulates into an fp32 C without residual");
  SD_CHECK(N % 128 == 0, "tcgen05 GEMM needs N % 128 == 0");
  SD_CHECK(K % 8 == 0, "tcgen05 GEMM needs K % 8 == 0 (16B TMA pitch)");
  SD_CHECK(epi >= 0 && epi <= 2, "unknown GEMM epilogue");
  SD_CHECK(!((resid || out_kind == 2) && epi != 0), "fp32 output / residual add only with the identity epilogue");
  SD_CHECK(!(resid && out_kind != 2), "a residual GEMM writes fp32");
  SD_CHECK(!ln_resid || (resid && ln_resid->stats && ln_resid->g && ln_resid->b), "LayerNorm-residual needs resid, stats and the affine");
  SD_CHECK(bias != nullptr, "bias required");
  SD_CHECK((a_fmt | 1) == 1 && out_kind >= 0 && out_kind <= 2, "bad operand format");
  // measured on B200: tcgen05.mma.kind::f16 with a_format != b_format faults as an illegal instruction
  SD_CHECK(a_fmt == w_fmt, "A and W must share one 16-bit format");
  int cfg = force_cfg;
  int ksplit = split_k;
  if (ksplit != 1 && !cfg) cfg = pick_cfg(M, N, K);  // the tuner replays launches on the caller's C: not idempotent under accumulation
  if (!cfg) {
    // First eager call of a (shape, epilogue) times every legal tile configuration on the caller's buffers and keeps the
    // fastest (the GEMM is idempotent unless C aliases an input); under stream capture, or with SEQDIFF_GEMM_TUNE=0, the
    // static cost model decides.  The sampling loop runs one un-captured forward before it captures its graph, so every
    // shape of the model is tuned by then.
    static const int tune = [] { const char* e = getenv("SEQDIFF_GEMM_TUNE"); return e ? atoi(e) : 1; }();
    static std::mutex mu;
    static std::unordered_map<uint64_t, int> tuned;
    const int rkind = resid ? (ln_resid ? 2 : 1) : 0;
    const uint64_t key = (static_cast<uint64_t>(M) << 40) ^ (static_cast<uint64_t>(N) << 24) ^ (static_cast<uint64_t>(K) << 8) ^
                         (static_cast<uint64_t>(epi) << 6) ^ (static_cast<uint64_t>(out_kind) << 4) ^ (static_cast<uint64_t>(rkind) << 2) ^
                         static_cast<uint64_t>(a_fmt);
    {
      std::lock_guard<std::mutex> g(mu);
      auto it = tuned.find(key);
      if (it != tuned.end()) cfg = it->second;
    }
    if (!cfg) {
      cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
      SD_CUDA(cudaStreamIsCapturing(s, &cap));
      const bool can_tune = tune && cap == cudaStreamCaptureStatusNone && M > 64 && C != A && C != static_cast<const void*>(resid);
      if (!can_tune) {
        cfg = pick_cfg(M, N, K);
      } else {
        // Candidates are timed the way the sampling loop runs them: 8 launches captured into a CUDA graph on a private
        // stream, replayed once to warm up and once between two events.  (Eager launches between events are dominated by
        // launch latency for these 10-30 us kernels and picked e.g. 256x384 pair tiles where 128x192 is 10 % faster in situ.)
        static cudaStream_t tune_streams[64] = {};  // one private stream per device (a process may hold handles on several GPUs)
        int dev_id = 0;
        SD_CUDA(cudaGetDevice(&dev_id));
        SD_CHECK(dev_id >= 0 && dev_id < 64, "device ordinal out of range");
        if (!tune_streams[dev_id]) SD_CUDA(cudaStreamCreateWithFlags(&tune_streams[dev_id], cudaStreamNonBlocking));
        cudaStream_t ts = tune_streams[dev_id];
        cudaEvent_t e0, e1;
        SD_CUDA(cudaEventCreate(&e0));
        SD_CUDA(cudaEventCreate(&e1));
        SD_CUDA(cudaStreamSynchronize(s));  // the operands are ready
        float best_ms = 0.f;
        constexpr int kReps = 8;
        for (int cand : {128, 192, 256, 128 | (1 << 16), 192 | (1 << 16), 256 | (1 << 16)}) {
          if (N % (cand & 0xffff)) continue;
          // eager warm-up launch: kernel attributes and the descriptor cache are set outside the capture
          SD_TRY(gemm_16(M, N, K, A, a_fmt, W, w_fmt, bias, resid, epi, C, out_kind, ts, cand, ln_resid));
          cudaGraph_t graph = nullptr;
          cudaGraphExec_t exec = nullptr;
          SD_CUDA(cudaStreamBeginCapture(ts, cudaStreamCaptureModeThreadLocal));
          int rc = SEQDIFF_OK;
          for (int r8 = 0; r8 < kReps && rc == SEQDIFF_OK; ++r8)
            rc = gemm_16(M, N, K, A, a_fmt, W, w_fmt, bias, resid, epi, C, out_kind, ts, cand, ln_resid);
          cudaError_t ce = cudaStreamEndCapture(ts, &graph);
          if (rc != SEQDIFF_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
          SD_CUDA(ce);
          ce = cudaGraphInstantiate(&exec, graph, 0);
          cudaGraphDestroy(graph);
          SD_CUDA(ce);
          float ms = 0.f;
          ce = cudaGraphLaunch(exec, ts);  // warm-up replay
          for (int rep = 0; rep < 3 && ce == cudaSuccess; ++rep) {  // best of three timed replays: one noisy sample flipped 128 / 192 / 256 picks between runs
            float ms1 = 0.f;
            ce = cudaEventRecord(e0, ts);
            if (ce == cudaSuccess) ce = cudaGraphLaunch(exec, ts);
            if (ce == cudaSuccess) ce = cudaEventRecord(e1, ts);
            if (ce == cudaSuccess) ce = cudaEventSynchronize(e1);
            if (ce == cudaSuccess) ce = cudaEventElapsedTime(&ms1, e0, e1);
            if (rep == 0 || ms1 < ms) ms = ms1;
          }
          cudaGraphExecDestroy(exec);
          SD_CUDA(ce);
          if (!cfg || ms < best_ms) { cfg = cand; best_ms = ms; }
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        SD_CUDA(cudaStreamSynchronize(ts));  // C holds the result of the last candidate before the caller's stream goes on
        std::lock_guard<std::mutex> g(mu);
        tuned[key] = cfg;
        // SEQDIFF_GEMM_TUNE_LOG=1: one line per tuned (shape, epilogue) -- which tile configurations the model's shapes really select
        static const bool tlog = [] { const char* e = getenv("SEQDIFF_GEMM_TUNE_LOG"); return e && e[0] == '1'; }();
        if (tlog) fprintf(stderr, "[seqdiff gemm tune] M=%d N=%d K=%d epi=%d out=%d resid=%d -> bn=%d cg2=%d (%.1f us)\n", M, N, K, epi, out_kind, rkind, cfg & 0xffff, cfg >> 16, best_ms * 1e3 / kReps);
        return SEQDIFF_OK;  // C already holds the result (every candidate wrote it)
      }
    }
  }
  const int bn = cfg & 0xffff;
  const bool cg2 = (cfg >> 16) != 0;
  SD_CHECK((bn == 128 || bn == 192 || bn == 256) && N % bn == 0, "bad tile width");
  CUtensorMap ta, tb;
  SD_TRY(make_tmap(A, a_fmt, M, K, kBM, &ta));
  SD_TRY(make_tmap(W, w_fmt, N, K, cg2 ? bn / 2 : bn, &tb));
  CUtensorMap tc = ta;  // store map of 16-bit outputs (unused for fp32 C)
  if (out_kind != 2) SD_TRY(make_tmap_store16(C, out_kind, M, N, &tc));
  const uint32_t idesc = umma_idesc_16(cg2 ? 2 * kBM : kBM, bn, static_cast<uint32_t>(a_fmt), static_cast<uint32_t>(w_fmt));
  if (ksplit != 1) {
    const int nkb = ceil_div(K, kBK);
    if (ksplit < 0) {  // auto: one scheduled tile per CTA slot, at least 4 k-blocks per k-range
      const int tiles = ceil_div(M, cg2 ? 2 * kBM : kBM) * (N / bn);
      const int slots = cg2 ? num_sms() / 2 : num_sms();
      ksplit = slots / tiles;
      if (ksplit > nkb / 4) ksplit = nkb / 4;
    }
    if (ksplit > nkb) ksplit = nkb;  // no more k-ranges than k-blocks
    if (ksplit < 1) ksplit = 1;
  }
#define SD_DISPATCH(BN_)                                                                                          \
  return cg2 ? dispatch_tc<BN_, true>(ta, tb, tc, bias, resid, epi, C, out_kind, M, N, K, idesc, s, ln_resid, ksplit) \
             : dispatch_tc<BN_, false>(ta, tb, tc, bias, resid, epi, C, out_kind, M, N, K, idesc, s, ln_resid, ksplit)
  if (bn == 256) { SD_DISPATCH(256); }
  if (bn == 192) { SD_DISPATCH(192); }
  SD_DISPATCH(128);
#undef SD_DISPATCH
}

// =====================================================================================================
// fp32 SIMT kernel (parity mode).  64x64 tile, BK=16, 256 threads x (4x4) outputs, fp32 FMA chain in k order.
// =====================================================================================================
template <int EPI, bool RESID>
__global__ void __launch_bounds__(256) gemm_f32_kernel(const float* __restrict__ A, const float* __restrict__ W,
                                                       const float* __restrict__ bias, const float* __restrict__ resid,
                                                       float* __restrict__ C, int M, int N, int K) {
  constexpr int TM = 64, TN = 64, TK = 16;
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  __shared__ float sA[TK][TM + 4];
  __shared__ float sW[TK][TN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  float acc[4][4] = {};
  const int lr = tid >> 2;        // 0..63 row inside the tile
  const int lk = (tid & 3) * 4;   // 0,4,8,12
  for (int k0 = 0; k0 < K; k0 += TK) {
    float4 a4 = make_float4(0, 0, 0, 0), w4 = make_float4(0, 0, 0, 0);
    const int ar = m0 + lr, wr = n0 + lr;
    if (k0 + lk + 3 < K) {
      if (ar < M) a4 = *reinterpret_cast<const float4*>(A + static_cast<size_t>(ar) * K + k0 + lk);
      if (wr < N) w4 = *reinterpret_cast<const float4*>(W + static_cast<size_t>(wr) * K + k0 + lk);
    } else {
      float ta[4] = {0, 0, 0, 0}, tw[4] = {0, 0, 0, 0};
      for (int t = 0; t < 4; ++t)
        if (k0 + lk + t < K) {
          if (ar < M) ta[t] = A[static_cast<size_t>(ar) * K + k0 + lk + t];
          if (wr < N) tw[t] = W[static_cast<size_t>(wr) * K + k0 + lk + t];
        }
      a4 = make_float4(ta[0], ta[1], ta[2], ta[3]);
      w4 = make_float4(tw[0], tw[1], tw[2], tw[3]);
    }
    sA[lk][lr] = a4.x; sA[lk + 1][lr] = a4.y; sA[lk + 2][lr] = a4.z; sA[lk + 3][lr] = a4.w;
    sW[lk][lr] = w4.x; sW[lk + 1][lr] = w4.y; sW[lk + 2][lr] = w4.z; sW[lk + 3][lr] = w4.w;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&sA[k][ty * 4]);
      const float4 w = *reinterpret_cast<const float4*>(&sW[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + ty * 4 + i;
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = n0 + tx * 4 + j;
      if (c >= N) continue;
      float v = acc[i][j] + bias[c];
      if (EPI == 1) v = gelu_erf(v);
      if (EPI == 2) v = silu(v);
      if (RESID) v += resid[static_cast<size_t>(r) * N + c];
      C[static_cast<size_t>(r) * N + c] = v;
    }
  }
}

int gemm_f32(int M, int N, int K, const float* A, const float* W, const float* bias, const float* resid, int epi, float* C,
             cudaStream_t s) {
  SD_CHECK(M > 0 && N > 0 && K > 0, "empty GEMM");
  SD_CHECK(K % 4 == 0, "fp32 GEMM needs K % 4 == 0");
  SD_CHECK(!(resid && epi != 0), "residual add is only fused with the identity epilogue");
  dim3 grid(ceil_div(N, 64), ceil_div(M, 64));
  if (resid) SD_CUDA(launch_k(gemm_f32_kernel<0, true>, dim3(grid), dim3(256), 0, s, A, W, bias, resid, C, M, N, K));
  else if (epi == 0) SD_CUDA(launch_k(gemm_f32_kernel<0, false>, dim3(grid), dim3(256), 0, s, A, W, bias, resid, C, M, N, K));
  else if (epi == 1) SD_CUDA(launch_k(gemm_f32_kernel<1, false>, dim3(grid), dim3(256), 0, s, A, W, bias, resid, C, M, N, K));
  else if (epi == 2) SD_CUDA(launch_k(gemm_f32_kernel<2, false>, dim3(grid), dim3(256), 0, s, A, W, bias, resid, C, M, N, K));
  else {
    set_error("unknown GEMM epilogue");
    return SEQDIFF_ERR_INVALID;
  }
  SD_LAUNCHED("gemm_f32", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
