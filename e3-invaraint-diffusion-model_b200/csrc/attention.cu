// attention.cu -- the 15 attention cores per forward (3 SELayer + 6 self + 6 cross), i.e. HF
// BertSelfAttention with transformers-4.38.2 `relative_key` semantics (SURVEY.md Appendix A):
//
//   S[l,r]  = ( q_l . k_r  +  q_l . E[l - r + P - 1] ) / 8  +  (1 - mask[r]) * -10000
//   out_l   = softmax_r(S[l,:]) @ V
//
// E = distance_embedding [2P-1, 64], shared by all heads; cross-attention has no E term.
//
// 16-bit kernel (bf16 or fp16 operands): one CTA per (query block of BQ rows, head, graph); each warp owns 16 query rows and runs
// m16n8k16 bf16 tensor-core MMAs with fp32 accumulation, flash-style online softmax over 128-key blocks.
// The relative term is a second MMA, QE = Q . Ewin^T, against the (BQ+128)-row window of E that this
// (query block, key block) pair can touch; warp w only needs window rows [16w, 16w+144).  QE is staged
// in a per-warp fp32 smem panel and added to S along the skewed diagonal j = l_local - r_local + 127
// (the "skewing" step; accumulator fragments cannot be shifted in registers).
// fp32 kernel (parity mode): one warp per query row, straight loops.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace seqdiff {

#ifdef SEQDIFF_AB_KERNELS  // legacy mma.sync kernel: A/B reference only (see attention_any16 below)
// ---------------------------------------------------------------------------------------------------
// small PTX helpers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;  // src-size 0 => 16 zero bytes written
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
template <typename T> __device__ __forceinline__ void mma_16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1);
template <> __device__ __forceinline__ void mma_16<bf16>(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <> __device__ __forceinline__ void mma_16<f16>(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// tiles are [rows][64 bf16] = 128 B rows; 16 B chunks XOR-swizzled by (row & 7) => ldmatrix is conflict-free
__device__ __forceinline__ uint32_t swz(int row, int chunk) { return static_cast<uint32_t>(row * 128 + ((chunk ^ (row & 7)) << 4)); }

constexpr int kKB = 128;     // keys per block
constexpr int kQEPitch = 148;  // floats per staged QE row (144 used)

template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }

// NBUF = 2 double-buffers the per-key-block tiles (K, V, E window, mask) so block kb+1 streams in under block kb's MMAs.
template <bool REL, int BQ, int NBUF> struct AttnSmem {
  static constexpr int kWarps = BQ / 16;
  static constexpr int kERows = BQ + 128;
  static constexpr int kBlk = 2 * kKB * 128 + (REL ? kERows * 128 : 0) + kKB * 4;  // K | V | E | mask, per buffer
  static constexpr int kQ = 0;
  static constexpr int kBuf = kQ + BQ * 128;
  static constexpr int kQE = kBuf + NBUF * kBlk;
  static constexpr int kBytes = kQE + (REL ? kWarps * 16 * kQEPitch * 4 : 0);
  static constexpr int kKOff = 0, kVOff = kKB * 128, kEOff = 2 * kKB * 128, kMOff = 2 * kKB * 128 + (REL ? kERows * 128 : 0);
};

template <typename T, bool REL, int BQ, int NBUF>
__global__ void __launch_bounds__(BQ * 2) attention_16_kernel(const T* __restrict__ q, int ldq, const T* __restrict__ k, int ldk,
                                                              const T* __restrict__ v, int ldv, const T* __restrict__ E, int P,
                                                              const float* __restrict__ key_mask, T* __restrict__ out, int heads,
                                                              int Lq, int Lk) {
  using SM = AttnSmem<REL, BQ, NBUF>;
  constexpr int NT = BQ * 2;
  constexpr int NG = REL ? 3 : 2;  // cp.async groups per key block: K, (E,) V -- consumed in that order
  constexpr float kScale2 = 0.125f * 1.44269504088896f;  // 1/sqrt(64) * log2(e): softmax runs in the log2 domain
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int q0 = blockIdx.x * BQ, h = blockIdx.y, b = blockIdx.z;

  const T* qb = q + (static_cast<size_t>(b) * Lq) * ldq + h * 64;
  const T* kb_ = k + (static_cast<size_t>(b) * Lk) * ldk + h * 64;
  const T* vb = v + (static_cast<size_t>(b) * Lk) * ldv + h * 64;
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access

  auto load_block = [&](int kb) {  // issues NG commit groups: {K (+Q on the first call)}, {E}, {V}
    const int k0 = kb * kKB;
    const uint32_t buf = sbase + SM::kBuf + (kb % NBUF) * SM::kBlk;
    for (int i = tid; i < kKB * 8; i += NT) {
      const int r = i >> 3, c = i & 7;
      const bool ok = k0 + r < Lk;
      cp_async16(buf + SM::kKOff + swz(r, c), kb_ + static_cast<size_t>(ok ? k0 + r : 0) * ldk + c * 8, ok);
    }
    cp_async_commit();
    if (REL) {
      const int ebase = q0 - k0 + P - 1 - 127;
      for (int i = tid; i < SM::kERows * 8; i += NT) {
        const int r = i >> 3, c = i & 7;
        const int idx = ebase + r;
        const bool ok = idx >= 0 && idx < 2 * P - 1;
        cp_async16(buf + SM::kEOff + swz(r, c), E + static_cast<size_t>(ok ? idx : 0) * 64 + c * 8, ok);
      }
      cp_async_commit();
    }
    for (int i = tid; i < kKB * 8; i += NT) {
      const int r = i >> 3, c = i & 7;
      const bool ok = k0 + r < Lk;
      cp_async16(buf + SM::kVOff + swz(r, c), vb + static_cast<size_t>(ok ? k0 + r : 0) * ldv + c * 8, ok);
    }
    cp_async_commit();
    float* sMask = reinterpret_cast<float*>(smem + SM::kBuf + (kb % NBUF) * SM::kBlk + SM::kMOff);
    for (int i = tid; i < kKB; i += NT) {
      const int r = k0 + i;
      // additive mask (1-m)*-10000 of the reference, pre-multiplied by log2(e); tile padding beyond Lk is excluded outright
      sMask[i] = (r < Lk) ? (1.0f - key_mask[static_cast<size_t>(b) * Lk + r]) * (-10000.0f * 1.44269504088896f) : -INFINITY;
    }
  };

  // ---- Q tile: rides in the first commit group together with K(0) ----
  for (int i = tid; i < BQ * 8; i += NT) {
    const int r = i >> 3, c = i & 7;
    const bool ok = q0 + r < Lq;
    cp_async16(sbase + SM::kQ + swz(r, c), qb + static_cast<size_t>(ok ? q0 + r : 0) * ldq + c * 8, ok);
  }
  load_block(0);

  // per-lane ldmatrix offsets, hoisted: every tile row offset used below is a multiple of 8 rows, so (row & 7) == (lane & 7)
  // and the swizzled 16 B chunk only depends on the k-step / d-pair -> the unrolled loops address smem as base + immediate.
  uint32_t offB[4], offV[4];
  {
    const int x7 = lane & 7;
    const int rowB = x7 + ((lane >> 4) << 3), hiB = (lane >> 3) & 1;  // B operand, [n][k] tiles (K, E)
    const int rowV = x7 + (((lane >> 3) & 1) << 3), hiV = lane >> 4;   // B operand via .trans, [k][n] tile (V)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      offB[i] = static_cast<uint32_t>(rowB * 128 + (((i * 2 + hiB) ^ x7) << 4));
      offV[i] = static_cast<uint32_t>(rowV * 128 + (((i * 2 + hiV) ^ x7) << 4));
    }
  }
  uint32_t qa[4][4];  // A fragments of this warp's 16 query rows, 4 k-steps
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};

  const int nkb = (Lk + kKB - 1) / kKB;
  for (int kb = 0; kb < nkb; ++kb) {
    const uint32_t buf = sbase + SM::kBuf + (kb % NBUF) * SM::kBlk;
    const float* sMask = reinterpret_cast<const float*>(smem + SM::kBuf + (kb % NBUF) * SM::kBlk + SM::kMOff);
    bool pref = false;
    if (NBUF == 2) {
      pref = kb + 1 < nkb;
      if (pref) load_block(kb + 1);  // other buffer: released by the barrier that ended iteration kb-1
    } else if (kb > 0) {
      load_block(kb);
    }
    // ---- K (and Q) landed? ----
    if (pref) cp_async_wait_group<NG - 1 + NG>(); else cp_async_wait_group<NG - 1>();
    __syncthreads();
    if (kb == 0) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)
        ldsm_x4(sbase + SM::kQ + swz(warp * 16 + (lane & 15), ks * 2 + (lane >> 4)), qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
    }

    // ---- S = Q K^T : 16 rows x 128 keys per warp ----
    float s[16][4];
#pragma unroll
    for (int i = 0; i < 16; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
    // k-step outer: 16 independent accumulators between two MMAs on the same one (HMMA latency hidden by ILP)
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
      for (int np = 0; np < 8; ++np) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(buf + SM::kKOff + np * 2048 + offB[ks], b0, b1, b2, b3);
        mma_16<T>(s[2 * np], qa[ks], b0, b1);
        mma_16<T>(s[2 * np + 1], qa[ks], b2, b3);
      }
    }

    if (REL) {
      if (pref) cp_async_wait_group<1 + NG>(); else cp_async_wait_group<1>();
      __syncthreads();
      // ---- QE = Q . Ewin[16w : 16w+144]^T, staged, then added along the skewed diagonal ----
      float* st = reinterpret_cast<float*>(smem + SM::kQE) + warp * 16 * kQEPitch;
      const uint32_t ebase_w = buf + SM::kEOff + warp * 2048;
      float* st0 = st + g * kQEPitch + 2 * t;
      float* st1 = st + (g + 8) * kQEPitch + 2 * t;
#pragma unroll
      for (int cg = 0; cg < 3; ++cg) {  // 3 groups of 3 x 16 window columns: 6 independent accumulators per k-step
        float e[6][4];
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) e[i][j] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
          for (int cc = 0; cc < 3; ++cc) {
            uint32_t b0, b1, b2, b3;
            ldsm_x4(ebase_w + (cg * 3 + cc) * 2048 + offB[ks], b0, b1, b2, b3);
            mma_16<T>(e[2 * cc], qa[ks], b0, b1);
            mma_16<T>(e[2 * cc + 1], qa[ks], b2, b3);
          }
        }
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) {
          const int col = (cg * 3 + cc) * 16;
          *reinterpret_cast<float2*>(st0 + col) = make_float2(e[2 * cc][0], e[2 * cc][1]);
          *reinterpret_cast<float2*>(st1 + col) = make_float2(e[2 * cc][2], e[2 * cc][3]);
          *reinterpret_cast<float2*>(st0 + col + 8) = make_float2(e[2 * cc + 1][0], e[2 * cc + 1][1]);
          *reinterpret_cast<float2*>(st1 + col + 8) = make_float2(e[2 * cc + 1][2], e[2 * cc + 1][3]);
        }
      }
      __syncwarp();
      // window-local column of E for (row i, key rl):  j' = i - rl + 127  in [0, 142]
      const float* r0p = st + g * kQEPitch + g + 127 - 2 * t;
      const float* r1p = st + (g + 8) * kQEPitch + g + 8 + 127 - 2 * t;
#pragma unroll
      for (int n = 0; n < 16; ++n) {
        s[n][0] += r0p[-8 * n];
        s[n][1] += r0p[-8 * n - 1];
        s[n][2] += r1p[-8 * n];
        s[n][3] += r1p[-8 * n - 1];
      }
      __syncwarp();
    }

    // ---- scale (after adding Rel), mask, online softmax in the log2 domain ----
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int n = 0; n < 16; ++n) {
      const float2 mk = *reinterpret_cast<const float2*>(sMask + n * 8 + 2 * t);
      s[n][0] = fmaf(s[n][0], kScale2, mk.x);
      s[n][1] = fmaf(s[n][1], kScale2, mk.y);
      s[n][2] = fmaf(s[n][2], kScale2, mk.x);
      s[n][3] = fmaf(s[n][3], kScale2, mk.y);
      mx[0] = fmaxf(mx[0], fmaxf(s[n][0], s[n][1]));
      mx[1] = fmaxf(mx[1], fmaxf(s[n][2], s[n][3]));
    }
    float corr[2], rs[2] = {0.f, 0.f};
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float m_new = fmaxf(m_run[r], mx[r]);
      corr[r] = (m_run[r] == -INFINITY) ? 0.f : ex2_approx(m_run[r] - m_new);
      m_run[r] = m_new;
    }
    uint32_t pa[8][4];  // P as 16-bit A fragments for P @ V
#pragma unroll
    for (int n = 0; n < 16; ++n) {
      const float p0 = ex2_approx(s[n][0] - m_run[0]), p1 = ex2_approx(s[n][1] - m_run[0]);
      const float p2 = ex2_approx(s[n][2] - m_run[1]), p3 = ex2_approx(s[n][3] - m_run[1]);
      rs[0] += p0 + p1;
      rs[1] += p2 + p3;
      pa[n >> 1][(n & 1) * 2 + 0] = pack2<T>(p0, p1);
      pa[n >> 1][(n & 1) * 2 + 1] = pack2<T>(p2, p3);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 1);
      rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 2);
      l_run[r] = l_run[r] * corr[r] + rs[r];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      o[i][0] *= corr[0]; o[i][1] *= corr[0];
      o[i][2] *= corr[1]; o[i][3] *= corr[1];
    }
    // ---- O += P V ----
    if (pref) cp_async_wait_group<NG>(); else cp_async_wait_group<0>();
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(buf + SM::kVOff + kk * 2048 + offV[dp], b0, b1, b2, b3);
        mma_16<T>(o[2 * dp], pa[kk], b0, b1);
        mma_16<T>(o[2 * dp + 1], pa[kk], b2, b3);
      }
    }
    if (kb + 1 < nkb) __syncthreads();  // every warp is done with this buffer before it is refilled
  }

  // ---- normalise and store ----
  const int H = heads * 64;
  const float inv0 = 1.0f / l_run[0], inv1 = 1.0f / l_run[1];
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const int col = h * 64 + n * 8 + 2 * t;
    if (r0 < Lq) *reinterpret_cast<uint32_t*>(out + (static_cast<size_t>(b) * Lq + r0) * H + col) = pack2<T>(o[n][0] * inv0, o[n][1] * inv0);
    if (r1 < Lq) *reinterpret_cast<uint32_t*>(out + (static_cast<size_t>(b) * Lq + r1) * H + col) = pack2<T>(o[n][2] * inv1, o[n][3] * inv1);
  }
}

template <typename T, bool REL, int BQ, int NBUF>
static int launch_attn_16(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* E,
                          int P, const float* mask, T* out, cudaStream_t s) {
  using SM = AttnSmem<REL, BQ, NBUF>;
  auto kfn = attention_16_kernel<T, REL, BQ, NBUF>;
  static bool configured = false;
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
    configured = true;
  }
  dim3 grid(ceil_div(Lq, BQ), heads, B);
  SD_CUDA(launch_k(kfn, dim3(grid), dim3(BQ * 2), SM::kBytes, s, q, ldq, k, ldk, v, ldv, E, P, mask, out, heads, Lq, Lk));
  SD_LAUNCHED(REL ? "attention_16_rel" : "attention_16_norel", s);
  return SEQDIFF_OK;
}

template <typename T>
static int attention_16(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv,
                        const T* dist_emb, int P, const float* key_mask, T* out, cudaStream_t s) {
  SD_CHECK(B > 0 && heads > 0 && Lq > 0 && Lk > 0, "empty attention");
  SD_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0, "row strides must be multiples of 8 elements");
  SD_CHECK(!dist_emb || (Lq <= P && Lk <= P), "sequence longer than max_position_embeddings");
  // One key block (Lk <= 128): BQ = 64, single buffer (~100 KB) -> two CTAs per SM overlap each other's fill and MMAs.
  // Several key blocks: BQ = 128 with double-buffered K/V/E (218 KB, one CTA per SM) -> the next block streams in under
  // the current block's MMAs and K/V/E are re-read half as often.  SEQDIFF_ATTN_CFG=64|128 forces a shape (tuning knob).
  static const int forced = [] { const char* e = getenv("SEQDIFF_ATTN_CFG"); return e ? atoi(e) : 0; }();
  const bool multi = forced ? forced == 128 : Lk > kKB;
#define SD_ATTN(REL_)                                                                                                         \
  return multi ? launch_attn_16<T, REL_, 128, 2>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s)     \
               : launch_attn_16<T, REL_, 64, 1>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s)
  if (dist_emb) { SD_ATTN(true); }
  SD_ATTN(false);
#undef SD_ATTN
}
#endif  // SEQDIFF_AB_KERNELS

// 16-bit modes: the persistent pipelined tcgen05 kernel (attention_pipe.cu) for every shape.  The two kernels it superseded --
// the one-item-per-CTA tcgen05 kernel (attention_tc.cu) and the mma.sync kernel above -- are A/B references only: they are
// compiled in when the library is built with SEQDIFF_AB_KERNELS=1 (build.py) and then selectable with SEQDIFF_ATTN = tc | mma.
#ifdef SEQDIFF_AB_KERNELS
static int attn_choice() {
  static const int v = [] {
    const char* e = getenv("SEQDIFF_ATTN");
    if (!e) return 0;
    const std::string c(e);
    return c == "tc" ? 1 : (c == "mma" ? 2 : (c == "auto_r1" ? 3 : 0));
  }();
  return v;
}
#endif
template <typename T>
static int attention_any16(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb,
                           int P, const float* key_mask, T* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
#ifdef SEQDIFF_AB_KERNELS
  const int c = attn_choice();
  if (c != 0 && !pack) {
    SD_CHECK(kv_div == 1, "the A/B reference attention kernels read the keys of their own graph only");
    // "auto_r1": the per-shape choice before the pipelined kernel existed (legacy for one-key-block relative_key, tc otherwise)
    const bool legacy = c == 2 || (c == 3 && dist_emb != nullptr && Lk <= kKB);
    if (legacy) return attention_16<T>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s);
    return attention_tc<T>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s);
  }
#endif
  return attention_pipe<T>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, kv_div);
}
template <>
int attention<bf16>(int B, int heads, int Lq, int Lk, const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv,
                    const bf16* dist_emb, int P, const float* key_mask, bf16* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
  return attention_any16<bf16>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, kv_div);
}
template <>
int attention<f16>(int B, int heads, int Lq, int Lk, const f16* q, int ldq, const f16* k, int ldk, const f16* v, int ldv,
                   const f16* dist_emb, int P, const float* key_mask, f16* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
  return attention_any16<f16>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, kv_div);
}

// ---------------------------------------------------------------------------------------------------
// fp32 parity kernel: one warp per query row; scores for the whole row live in smem.  Query graph b reads key graph b / kv_div.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) attention_f32_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ k, int ldk,
                                                            const float* __restrict__ v, int ldv, const float* __restrict__ E, int P,
                                                            const float* __restrict__ key_mask, float* __restrict__ out, int heads,
                                                            int Lq, int Lk, int kv_div) {
  extern __shared__ float sm[];
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* sq = sm + warp * 64;
  float* sc = sm + 8 * 64 + warp * Lk;
  const int l = blockIdx.x * 8 + warp, h = blockIdx.y, b = blockIdx.z, kg = b / kv_div;
  if (l >= Lq) return;
  const float* qrow = q + (static_cast<size_t>(b) * Lq + l) * ldq + h * 64;
  sq[lane] = qrow[lane];
  sq[lane + 32] = qrow[lane + 32];
  __syncwarp();
  float mx = -INFINITY;
  for (int r = lane; r < Lk; r += 32) {
    const float* kr = k + (static_cast<size_t>(kg) * Lk + r) * ldk + h * 64;
    float acc = 0.f, rel = 0.f;
#pragma unroll 4
    for (int d = 0; d < 64; d += 4) {
      const float4 kk = *reinterpret_cast<const float4*>(kr + d);
      acc = fmaf(sq[d], kk.x, acc); acc = fmaf(sq[d + 1], kk.y, acc);
      acc = fmaf(sq[d + 2], kk.z, acc); acc = fmaf(sq[d + 3], kk.w, acc);
    }
    if (E) {
      const float* er = E + static_cast<size_t>(l - r + P - 1) * 64;
#pragma unroll 4
      for (int d = 0; d < 64; d += 4) {
        const float4 ee = *reinterpret_cast<const float4*>(er + d);
        rel = fmaf(sq[d], ee.x, rel); rel = fmaf(sq[d + 1], ee.y, rel);
        rel = fmaf(sq[d + 2], ee.z, rel); rel = fmaf(sq[d + 3], ee.w, rel);
      }
    }
    const float sv = (acc + rel) / 8.0f + (1.0f - key_mask[static_cast<size_t>(kg) * Lk + r]) * -10000.0f;
    sc[r] = sv;
    mx = fmaxf(mx, sv);
  }
  mx = warp_max(mx);
  float sum = 0.f;
  for (int r = lane; r < Lk; r += 32) {
    const float e = expf(sc[r] - mx);
    sc[r] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  __syncwarp();
  float a0 = 0.f, a1 = 0.f;
  for (int r = 0; r < Lk; ++r) {
    const float p = sc[r] / sum;
    const float* vr = v + (static_cast<size_t>(kg) * Lk + r) * ldv + h * 64;
    a0 = fmaf(p, vr[lane], a0);
    a1 = fmaf(p, vr[lane + 32], a1);
  }
  float* orow = out + (static_cast<size_t>(b) * Lq + l) * (heads * 64) + h * 64;
  orow[lane] = a0;
  orow[lane + 32] = a1;
}

template <>
int attention<float>(int B, int heads, int Lq, int Lk, const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                     const float* dist_emb, int P, const float* key_mask, float* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
  SD_CHECK(pack == nullptr, "packed batches run in the 16-bit modes only");
  SD_CHECK(B > 0 && heads > 0 && Lq > 0 && Lk > 0, "empty attention");
  SD_CHECK(kv_div >= 1 && B % kv_div == 0, "every key graph must serve kv_div whole query graphs");
  SD_CHECK(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0, "row strides must be multiples of 4 elements");
  SD_CHECK(!dist_emb || (Lq <= P && Lk <= P), "sequence longer than max_position_embeddings");
  const size_t smem = (8 * 64 + 8 * static_cast<size_t>(Lk)) * sizeof(float);
  SD_CHECK(smem <= 48 * 1024, "fp32 attention: Lk too large");
  dim3 grid(ceil_div(Lq, 8), heads, B);
  SD_CUDA(launch_k(attention_f32_kernel, dim3(grid), dim3(256), smem, s, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, heads, Lq, Lk, kv_div));
  SD_LAUNCHED("attention_f32", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
