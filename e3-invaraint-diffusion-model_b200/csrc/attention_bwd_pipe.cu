// attention_bwd_pipe.cu -- backward of the attention core on tcgen05 (training step, BASELINE configs[3]); same math and interface as
// attention_train_tc.cu (nvcuda::wmma, 20 % issue utilisation at 8 warps per SM: 31 % of the training step) and attention_train.cu (fp32 SIMT,
// the parity reference).  Replaces what autograd derives for HF BertSelfAttention (SURVEY.md Appendix A) incl. the attention-
// probability dropout; reference call sites sequence_model/model.py:61 and 226-231.
//
// One work item = one (graph, head) with Lq, Lk <= 128: every product of the backward is a single 128-row UMMA tile.
//     phase 1 (tensor core)   S  = Q K^T                     dP~ = dO V^T                                  -> TMEM
//     phase 2 (CUDA cores)    P  = softmax(S / 8 + mask)     keep = Philox dropout mask (regenerated)
//                             D  = rowsum(P * keep * dP~)    dS = P * (keep * dP~ - D) / 8
//                             drop(P) = P * keep and dS -> shared memory, 16-bit, [query][key] rows of 128 B (SW128)
//     phase 3 (tensor core)   dQ = dS K                      dV = drop(P)^T dO          dK = dS^T Q        -> TMEM
//     phase 4 (CUDA cores)    TMEM -> 16-bit -> global (rows past the graph's lengths are not written)
// The [query][key] tiles written in phase 2 are read twice in phase 3: K-major as the A operand of dS K, and MN-major as the A
// operand of the two transposed products (the same bytes: an MN-major SW128 operand is exactly a [k][mn] tile with 128 B rows).
// Q, K, V, dO arrive by TMA and serve as K-major operands in phase 1 and as MN-major B operands in phase 3 -- nothing is
// transposed and nothing of size L x L touches HBM.
// Roles as in attention_pipe.cu: warp 0 TMA producer (operands of item i+1 are in flight while item i is processed), warp 1
// MMA issuer (phase 1 of item i+1 is issued right behind phase 3 of item i, i.e. under item i's epilogue), warps 2..9 two
// threads per row (64 keys each) for phases 2 and 4.
// relative_key (REL: self-attention with the distance embedding E, S[l,r] += q_l . E[l - r + P - 1]): with W = the 256-row window of E
// that a 128 x 128 item can touch (window row w <-> E row w + P - 128),
//     phase 1   QE = Q W^T [128 x 256] next to S; the relative term of key r is QE[l, l + 127 - r] (register barrel shift, as in
//               attention_pipe.cu); dP~ is issued into the S columns once S has been drained (TMEM: S|dP~ 128 + QE 256 + dE 128)
//     phase 3b  dSk[l, l + 127 - r] = dS[l, r] -- the skewed copy of dS, written over the P | dS tiles once the products that read
//               them have completed -- then  dQ += dSk W  and  dE_w += dSk^T Q  (two 128-row UMMAs; dE accumulates in TMEM over ALL
//               items of the CTA and is flushed once, with atomics, at the end).
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"
#include "skew.cuh"

namespace seqdiff {

namespace {
constexpr int kBT = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 elementwise
constexpr float kL2e = 1.44269504088896f;

template <bool REL> struct BwdSmem {
  static constexpr int kStages = REL ? 1 : 2;      // REL: the window of E and the skewed tile take the second stage's room
  static constexpr int kIn = 0;                    // kStages x (Q | K | V | dO), each [128][64] 16-bit SW128 = 16 KB
  static constexpr int kE = kIn + kStages * 4 * 16384;  // REL: [256 window rows][64], loaded once per CTA
  static constexpr int kP = kE + (REL ? 32768 : 0);     // drop(P): 2 tiles [128 q][64 keys]
  static constexpr int kdS = kP + 32768;           // dS: 2 tiles.  REL phase 3b: P | dS are overwritten by dSk = 4 tiles [128 q][64 window cols]
  static constexpr int kXch = kdS + 32768;         // [3 exchanges][2 halves][128] fp32
  static constexpr int kMask = kXch + 3 * 2 * 128 * 4;  // [128] additive mask (log2 domain)
  static constexpr int kBar = kMask + 128 * 4;
  static constexpr int kBytes = kBar + 256 + 1024;
};
// TMEM columns.  no-REL: S | dP~ | dQ | dV | dK side by side (phase 1 of item i+1 runs under the epilogue of item i).
// REL: S and dP~ share [0,128), QE [128,384) is reused by the outputs, dE [384,512) lives across items.
template <bool REL> struct BwdCols {
  static constexpr int kS = 0, kdP = REL ? 0 : 128, kQE = 128;
  static constexpr int kdQ = REL ? 128 : 256, kdV = REL ? 192 : 320, kdK = REL ? 256 : 384, kdE = 384;
};

__device__ __forceinline__ void ew_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
}  // namespace

template <typename T, bool REL>
__global__ void __launch_bounds__(kBT, 1)
attention_bwd_pipe_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                          const __grid_constant__ CUtensorMap tmdO, const __grid_constant__ CUtensorMap tmE, const float* __restrict__ key_mask, int heads,
                          int Lq, int Lk, int P, uint32_t fmt, int n_items, const DropSpec dr, T* __restrict__ dq, int lddq, T* __restrict__ dk, int lddk,
                          T* __restrict__ dv, int lddv, float* __restrict__ dE, const uint32_t* __restrict__ keep_in) {
  using BwdSmem = seqdiff::BwdSmem<REL>;
  using C = BwdCols<REL>;
  constexpr int kColS = C::kS, kColdP = C::kdP, kColdQ = C::kdQ, kColdV = C::kdV, kColdK = C::kdK;
  constexpr int NST = BwdSmem::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BwdSmem::kBar);
  uint64_t* in_full = bars;       // [2]
  uint64_t* in_empty = bars + 2;  // [2]
  uint64_t* s_full = bars + 4;
  uint64_t* s_empty = bars + 5;
  uint64_t* p_ready = bars + 6;
  uint64_t* o_full = bars + 7;
  uint64_t* o_empty = bars + 8;
  uint64_t* s_drained = bars + 9;   // REL: S + QE are in registers -> dP~ may be issued into the S columns
  uint64_t* dp_full = bars + 10;    // REL
  uint64_t* a_done = bars + 11;     // REL: the products that read the P | dS tiles have completed -> dSk may overwrite them
  uint64_t* sk_ready = bars + 12;   // REL
  uint64_t* e_full = bars + 13;     // REL: the window of E has landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);
  float* xch = reinterpret_cast<float*>(smem + BwdSmem::kXch);
  float* sMask = reinterpret_cast<float*>(smem + BwdSmem::kMask);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = warp_id_uniform();
  const int my_items = (static_cast<int>(blockIdx.x) < n_items) ? (n_items - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;

  if (tid == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmdO);
    for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
    mbar_init(s_full, 1);
    mbar_init(s_empty, 8);
    mbar_init(p_ready, 8);
    mbar_init(o_full, 1);
    mbar_init(o_empty, 8);
    mbar_init(s_drained, 8);
    mbar_init(dp_full, 1);
    mbar_init(a_done, 1);
    mbar_init(sk_ready, 8);
    mbar_init(e_full, 1);
    if (REL) tma_prefetch_desc(&tmE);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------ TMA producer ------------------------------------------
    if (REL && my_items > 0) {  // window row w <-> E row w + P - 128 (rows outside the table are zero-filled)
      mbar_expect_tx_e(e_full, 32768);
      tma_load_2d_e(smem + BwdSmem::kE, &tmE, e_full, 0, P - 128);
    }
    for (int i = 0; i < my_items; ++i) {
      const int item = static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
      const int h = item % heads, b = item / heads;
      const int st = i % NST;
      mbar_wait(&in_empty[st], ((i / NST) & 1) ^ 1);
      mbar_expect_tx_e(&in_full[st], 4 * 16384);
      uint8_t* base = smem + BwdSmem::kIn + st * 65536;
      tma_load_2d_e(base, &tmQ, &in_full[st], h * 64, b * Lq);
      tma_load_2d_e(base + 16384, &tmK, &in_full[st], h * 64, b * Lk);
      tma_load_2d_e(base + 32768, &tmV, &in_full[st], h * 64, b * Lk);
      tma_load_2d_e(base + 49152, &tmdO, &in_full[st], h * 64, b * Lq);
    }
  } else if (warp == 1) {
    // ------------------------------------------ MMA issuer --------------------------------------------
    const uint32_t idesc_s = umma_idesc_16(128, 128, fmt, fmt);                                    // A, B K-major
    const uint32_t idesc_e = umma_idesc_16(128, 256, fmt, fmt);                                    // QE = Q W^T
    const uint32_t idesc_q = umma_idesc_16(128, 64, fmt, fmt) | kUmmaBMnMajor;                     // dQ = dS K: A K-major, B = K MN-major
    const uint32_t idesc_t = umma_idesc_16(128, 64, fmt, fmt) | kUmmaAMnMajor | kUmmaBMnMajor;     // dV, dK, dE: A^T products
    auto stage_base = [&](int i) { return smem_u32(smem + BwdSmem::kIn + (i % NST) * 65536); };
    auto phase1 = [&](int i) {
      const int st = i % NST;
      mbar_wait(&in_full[st], (i / NST) & 1);
      if (REL) mbar_wait(o_empty, (i & 1) ^ 1);  // REL: QE lands on the columns the previous item's outputs were read from
      else mbar_wait(s_empty, (i & 1) ^ 1);      // the elementwise threads have drained S / dP of item i-1
      tc_fence_after();
      const uint32_t qa = stage_base(i), ka = qa + 16384, va = qa + 32768, oa = qa + 49152;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        umma_bf16_e(tmem_base + kColS, umma_desc_kmajor_sw128(qa + k * 32), umma_desc_kmajor_sw128(ka + k * 32), idesc_s, k ? 1u : 0u);
      if (REL) {
        if (i == 0) { mbar_wait(e_full, 0); tc_fence_after(); }
        const uint32_t ea = smem_u32(smem + BwdSmem::kE);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_e(tmem_base + C::kQE, umma_desc_kmajor_sw128(qa + k * 32), umma_desc_kmajor_sw128(ea + k * 32), idesc_e, k ? 1u : 0u);
        umma_commit_e(s_full);
        mbar_wait(s_drained, i & 1);  // S is in registers: dP~ reuses its columns
        tc_fence_after();
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        umma_bf16_e(tmem_base + kColdP, umma_desc_kmajor_sw128(oa + k * 32), umma_desc_kmajor_sw128(va + k * 32), idesc_s, k ? 1u : 0u);
      if (REL) umma_commit_e(dp_full); else umma_commit_e(s_full);
    };
    if (my_items > 0) phase1(0);
    for (int i = 0; i < my_items; ++i) {
      const int st = i % NST;
      mbar_wait(p_ready, i & 1);
      if (!REL) mbar_wait(o_empty, (i & 1) ^ 1);  // the epilogue of item i-1 has read its outputs (REL: waited for in phase 1)
      tc_fence_after();
      const uint32_t qa = stage_base(i), ka = qa + 16384, oa = qa + 49152;
      const uint32_t pa = smem_u32(smem + BwdSmem::kP), sa = smem_u32(smem + BwdSmem::kdS);
#pragma unroll
      for (int k = 0; k < 8; ++k)  // dQ[q, d] = sum_key dS[q, key] K[key, d]: k-step = 16 keys
        umma_bf16_e(tmem_base + kColdQ, umma_desc_kmajor_sw128(sa + (k >> 2) * 16384 + (k & 3) * 32), umma_desc_mnmajor_sw128(ka + k * 2048, 16384), idesc_q,
                    k ? 1u : 0u);
#pragma unroll
      for (int k = 0; k < 8; ++k)  // dV[key, d] = sum_q drop(P)[q, key] dO[q, d]: k-step = 16 queries; A = P^T: MN blocks = the two key tiles
        umma_bf16_e(tmem_base + kColdV, umma_desc_mnmajor_sw128(pa + k * 2048, 16384), umma_desc_mnmajor_sw128(oa + k * 2048, 16384), idesc_t, k ? 1u : 0u);
#pragma unroll
      for (int k = 0; k < 8; ++k)  // dK[key, d] = sum_q dS[q, key] Q[q, d]
        umma_bf16_e(tmem_base + kColdK, umma_desc_mnmajor_sw128(sa + k * 2048, 16384), umma_desc_mnmajor_sw128(qa + k * 2048, 16384), idesc_t, k ? 1u : 0u);
      if (REL) {
        umma_commit_e(a_done);
        mbar_wait(sk_ready, i & 1);  // dSk (4 tiles [128 q][64 window cols]) now occupies the P | dS tiles
        tc_fence_after();
        const uint32_t ea = smem_u32(smem + BwdSmem::kE);
#pragma unroll
        for (int k = 0; k < 16; ++k)  // dQ[q, d] += sum_w dSk[q, w] W[w, d]: k-step = 16 window rows
          umma_bf16_e(tmem_base + kColdQ, umma_desc_kmajor_sw128(pa + (k >> 2) * 16384 + (k & 3) * 32), umma_desc_mnmajor_sw128(ea + k * 2048, 16384), idesc_q, 1u);
#pragma unroll
        for (int half = 0; half < 2; ++half)  // dE_w[w, d] += sum_q dSk[q, w] Q[q, d], window rows 128 half .. + 127; accumulates over the CTA's items
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16_e(tmem_base + C::kdE + half * 64, umma_desc_mnmajor_sw128(pa + half * 32768 + k * 2048, 16384), umma_desc_mnmajor_sw128(qa + k * 2048, 16384),
                        idesc_t, (i | k) ? 1u : 0u);
      }
      umma_commit_e(o_full);
      umma_commit_e(&in_empty[st]);
      if (i + 1 < my_items) phase1(i + 1);
    }
  } else {
    // ------------------------------------------ elementwise threads -----------------------------------
    const int st_ = tid - 64;         // 0..255
    const int wq = warp & 3;          // TMEM lane quarter of this warp
    const int hf = (warp - 2) >> 2;   // key half (phase 2) / column half of the 64 output columns (phase 4)
    const int row = wq * 32 + lane;   // TMEM lane: query row in phases 1-2, key row for dV / dK in phase 4
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(wq * 32) << 16);
    const uint32_t thr = dr.p > 0.f ? static_cast<uint32_t>(static_cast<double>(dr.p) * 4294967296.0) : 0u;
    const float sc = dr.p > 0.f ? 1.0f / (1.0f - dr.p) : 1.0f;
    constexpr float kScale2 = 0.125f * kL2e;
    for (int i = 0; i < my_items; ++i) {
      const int item = static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
      const int h = item % heads, b = item / heads;
      if (st_ < 128) sMask[st_] = st_ < Lk ? (1.0f - __ldg(key_mask + static_cast<size_t>(b) * Lk + st_)) * (-10000.0f * kL2e) : -INFINITY;
      ew_bar();
      mbar_wait(s_full, i & 1);
      tc_fence_after();
      const bool live = row < Lq;
      // ---- P of (row, key half) ----
      float p[64];
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t x0[32], x1[32];
        if (REL) {
          // keys r of chunk kc = 2 hf + c pair with window columns w = row + 127 - r: for the warp's 32 rows that is the 2-chunk band of QE
          // starting at chunk qc0 = wq - kc + 3, and with X = those 64 columns of this lane's row, QE[row, w(r)] = X[lane + 31 - (r - 32 kc)]
          // (the barrel shift of attention_pipe.cu)
          const int qc0 = wq - (2 * hf + c) + 3;
          tmem_ld_32x32(t_lane + C::kQE + qc0 * 32, x0);
          tmem_ld_32x32(t_lane + C::kQE + (qc0 + 1) * 32, x1);
          tmem_ld_wait();
          const uint32_t ul = static_cast<uint32_t>(lane);
          shift_stage<16>(x0, x1, ul & 16u);
          shift_stage<8>(x0, x1, ul & 8u);
          shift_stage<4>(x0, x1, ul & 4u);
          shift_stage<2>(x0, x1, ul & 2u);
          shift_stage<1>(x0, x1, ul & 1u);
        }
        uint32_t r[32];
        tmem_ld_32x32(t_lane + kColS + hf * 64 + c * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float sv = __uint_as_float(r[j]);
          if (REL) sv += __uint_as_float(x0[31 - j]);
          sv = fmaf(sv, kScale2, sMask[hf * 64 + c * 32 + j]);
          p[c * 32 + j] = sv;
          mx = fmaxf(mx, sv);
        }
      }
      if (REL) {  // S and QE are in registers: dP~ may be issued into the S columns
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_drained);
      }
      xch[(0 * 2 + hf) * 128 + row] = mx;
      ew_bar();
      mx = fmaxf(mx, xch[(0 * 2 + (hf ^ 1)) * 128 + row]);
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < 64; ++j) {
        p[j] = ex2_approx(p[j] - mx);  // keys >= Lk carry -inf -> 0 (key 0 is always in range: mx is finite)
        sum += p[j];
      }
      xch[(1 * 2 + hf) * 128 + row] = sum;
      ew_bar();
      sum += xch[(1 * 2 + (hf ^ 1)) * 128 + row];
      const float inv = live ? 1.0f / sum : 0.f;  // rows past the graph's length contribute nothing to dK / dV
      // ---- dropout mask of this thread's 64 keys: one bit per key (regenerated from the forward's Philox stream) ----
      uint64_t keepbits = ~0ull;
      if (dr.p > 0.f && keep_in) {  // the forward kernel left the mask as bits: chunks 2 hf and 2 hf + 1 of this row
        const uint2 kb2 = __ldg(reinterpret_cast<const uint2*>(keep_in + ((static_cast<size_t>(b) * heads + h) * 128 + row) * 4 + 2 * hf));
        keepbits = static_cast<uint64_t>(kb2.x) | (static_cast<uint64_t>(kb2.y) << 32);
      } else if (dr.p > 0.f) {
        keepbits = 0ull;
        const size_t e_row = ((static_cast<size_t>(b) * heads + h) * Lq + row) * Lk + 64 * hf;
#pragma unroll
        for (int j4 = 0; j4 < 16; ++j4) {
          const uint64_t qd = (e_row + 4 * j4) >> 2;
          uint32_t w4[4] = {static_cast<uint32_t>(qd), static_cast<uint32_t>(qd >> 32), dr.site, dr.step};
          philox4x32_10(w4, static_cast<uint32_t>(dr.seed), static_cast<uint32_t>(dr.seed >> 32));
#pragma unroll
          for (int u = 0; u < 4; ++u) keepbits |= static_cast<uint64_t>(w4[u] >= thr ? 1u : 0u) << (4 * j4 + u);
        }
      }
      if (REL) {
        mbar_wait(dp_full, i & 1);
        tc_fence_after();
      }
      // ---- D = sum_key P keep dP~ ----
      float dsum = 0.f;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(t_lane + kColdP + hf * 64 + c * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          p[c * 32 + j] *= inv;
          const float kp = ((keepbits >> (c * 32 + j)) & 1ull) ? sc : 0.f;
          dsum = fmaf(p[c * 32 + j] * kp, __uint_as_float(r[j]), dsum);
        }
      }
      xch[(2 * 2 + hf) * 128 + row] = dsum;
      ew_bar();
      dsum += xch[(2 * 2 + (hf ^ 1)) * 128 + row];
      // ---- dS, drop(P) -> shared memory (tile hf, row `row`: 128 B = 8 chunks of 16 B, XOR-swizzled by row & 7) ----
      uint8_t* prow = smem + BwdSmem::kP + hf * 16384 + row * 128;
      uint8_t* srow = smem + BwdSmem::kdS + hf * 16384 + row * 128;
      uint32_t ds_keep[REL ? 32 : 1];  // REL: this thread's 64 dS values (16-bit pairs) for the skewed copy
      (void)ds_keep;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(t_lane + kColdP + hf * 64 + c * 32, r);
        tmem_ld_wait();
        uint32_t pp[16], ds[16];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float k0 = ((keepbits >> (c * 32 + j)) & 1ull) ? sc : 0.f, k1 = ((keepbits >> (c * 32 + j + 1)) & 1ull) ? sc : 0.f;
          const float p0 = p[c * 32 + j], p1 = p[c * 32 + j + 1];
          pp[j >> 1] = pack2<T>(p0 * k0, p1 * k1);
          ds[j >> 1] = pack2<T>(p0 * (__uint_as_float(r[j]) * k0 - dsum) * 0.125f, p1 * (__uint_as_float(r[j + 1]) * k1 - dsum) * 0.125f);
          if (REL) ds_keep[c * 16 + (j >> 1)] = ds[j >> 1];
        }
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
          const int chunk = ((c * 4 + qd) ^ (row & 7)) << 4;
          *reinterpret_cast<uint4*>(prow + chunk) = make_uint4(pp[4 * qd], pp[4 * qd + 1], pp[4 * qd + 2], pp[4 * qd + 3]);
          *reinterpret_cast<uint4*>(srow + chunk) = make_uint4(ds[4 * qd], ds[4 * qd + 1], ds[4 * qd + 2], ds[4 * qd + 3]);
        }
      }
      // S / dP are in registers / shared memory now: phase 1 of the next item may overwrite them
      tc_fence_before();
      fence_proxy_async_smem();  // generic-proxy writes (P, dS) -> visible to the tensor core
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(s_empty);
        mbar_arrive(p_ready);
      }
      if (REL) {
        // ---- phase 3b: dSk[l, l + 127 - r] = dS[l, r] over the P | dS tiles (4 tiles [128 q][64 window cols], SW128 K-major) ----
        mbar_wait(a_done, i & 1);  // dQ (first part), dV, dK have read P and dS
        uint8_t* skb = smem + BwdSmem::kP;
#pragma unroll
        for (int z = 0; z < 16; ++z) *reinterpret_cast<uint4*>(skb + (z * 256 + st_) * 16) = make_uint4(0u, 0u, 0u, 0u);
        ew_bar();
        uint8_t* skrow = skb + row * 128;
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const int w = row + 127 - (64 * hf + j);  // 0 .. 254
          const uint32_t pair = ds_keep[j >> 1];
          const uint16_t val = static_cast<uint16_t>((j & 1) ? (pair >> 16) : (pair & 0xffffu));
          *reinterpret_cast<uint16_t*>(skrow + (w >> 6) * 16384 + (((((w & 63) >> 3) ^ (row & 7))) << 4) + (w & 7) * 2) = val;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(sk_ready);
      }
      // ---- phase 4: outputs ----
      mbar_wait(o_full, i & 1);
      tc_fence_after();
      auto store_rows = [&](int col0, T* dst_base, int ld, int n_rows, int L) {
        uint32_t r[32];
        tmem_ld_32x32(t_lane + col0 + hf * 32, r);
        tmem_ld_wait();
        if (row < n_rows) {
          T* dst = dst_base + (static_cast<size_t>(b) * L + row) * ld + h * 64 + hf * 32;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<uint4*>(dst + 8 * j) =
                make_uint4(pack2<T>(__uint_as_float(r[8 * j]), __uint_as_float(r[8 * j + 1])), pack2<T>(__uint_as_float(r[8 * j + 2]), __uint_as_float(r[8 * j + 3])),
                           pack2<T>(__uint_as_float(r[8 * j + 4]), __uint_as_float(r[8 * j + 5])), pack2<T>(__uint_as_float(r[8 * j + 6]), __uint_as_float(r[8 * j + 7])));
        }
      };
      store_rows(kColdQ, dq, lddq, Lq, Lq);
      store_rows(kColdV, dv, lddv, Lk, Lk);
      store_rows(kColdK, dk, lddk, Lk, Lk);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
    }
    if (REL && my_items > 0) {
      // dE of the window rows, accumulated in TMEM over this CTA's items (complete: the last o_full covered it) -> E rows w + P - 128
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t r[32];
        tmem_ld_32x32(t_lane + C::kdE + half * 64 + hf * 32, r);
        tmem_ld_wait();
        const int j = half * 128 + row + P - 128;
        if (j >= 0 && j < 2 * P - 1) {
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            const float x = __uint_as_float(r[c]);
            if (x != 0.f) atomicAdd(dE + static_cast<size_t>(j) * 64 + hf * 32 + c, x);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <typename T> struct BwdFmt;
template <> struct BwdFmt<f16> { static constexpr int v = 0; };
template <> struct BwdFmt<bf16> { static constexpr int v = 1; };

// usable(...) = the shapes this kernel covers; everything else stays on attention_bwd_tc (wmma)
bool attention_bwd_pipe_usable(int Lq, int Lk, const void* dist_emb, float p_drop) {
  (void)dist_emb;
  return Lq <= 128 && Lk <= 128 && Lq >= 1 && Lk >= 1 && (p_drop <= 0.f || Lk % 4 == 0);
}

template <typename T, bool REL>
static int launch_bwd_pipe(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* E, int P,
                           const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s,
                           const uint32_t* keep_in) {
  SD_CHECK(B > 0 && heads > 0 && Lq >= 1 && Lk >= 1 && Lq <= 128 && Lk <= 128, "attention_bwd_pipe: one 128-row tile per (graph, head)");
  SD_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && lddq % 8 == 0 && lddk % 8 == 0 && lddv % 8 == 0, "row strides must be multiples of 8 elements");
  SD_CHECK(dr.p <= 0.f || Lk % 4 == 0, "dropout: Lk must be a multiple of 4");
  SD_CHECK(dout && dq && dk && dv && key_mask, "attention_bwd_pipe: null argument");
  SD_CHECK(!REL || (E && dE && Lq <= P && Lk <= P), "relative_key: needs the distance embedding, its gradient buffer and L <= max_position_embeddings");
  auto kfn = attention_bwd_pipe_kernel<T, REL>;
  using Sm = BwdSmem<REL>;
  static bool configured = false;
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Sm::kBytes));
    configured = true;
  }
  constexpr int fmt = BwdFmt<T>::v;
  CUtensorMap tq, tk, tv, to;
  SD_TRY(make_tmap(q, fmt, B * Lq, ldq, 128, &tq));
  SD_TRY(make_tmap(k, fmt, B * Lk, ldk, 128, &tk));
  SD_TRY(make_tmap(v, fmt, B * Lk, ldv, 128, &tv));
  SD_TRY(make_tmap(dout, fmt, B * Lq, heads * 64, 128, &to));
  CUtensorMap te = tq;
  if (REL) SD_TRY(make_tmap(E, fmt, 2 * P - 1, 64, 256, &te));
  const int n_items = B * heads;
  const int grid = n_items < num_sms() ? n_items : num_sms();
  SD_CUDA(launch_k(kfn, dim3(grid), dim3(kBT), Sm::kBytes, s, tq, tk, tv, to, te, key_mask, heads, Lq, Lk, P, static_cast<uint32_t>(fmt), n_items, dr, dq, lddq,
                   dk, lddk, dv, lddv, dE, keep_in));
  SD_LAUNCHED(REL ? "attention_bwd_pipe_rel" : "attention_bwd_pipe", s);
  return SEQDIFF_OK;
}
template <typename T>
int attention_bwd_pipe(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                       const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s,
                       const uint32_t* keep_in) {
  if (dist_emb)
    return launch_bwd_pipe<T, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, dout, dq, lddq, dk, lddk, dv, lddv, dE, s, keep_in);
  return launch_bwd_pipe<T, false>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, dout, dq, lddq, dk, lddk, dv, lddv, dE, s, keep_in);
}
template int attention_bwd_pipe<bf16>(int, int, int, int, const bf16*, int, const bf16*, int, const bf16*, int, const bf16*, int, const float*, DropSpec,
                                      const bf16*, bf16*, int, bf16*, int, bf16*, int, float*, cudaStream_t, const uint32_t*);
template int attention_bwd_pipe<f16>(int, int, int, int, const f16*, int, const f16*, int, const f16*, int, const f16*, int, const float*, DropSpec, const f16*,
                                     f16*, int, f16*, int, f16*, int, float*, cudaStream_t, const uint32_t*);

}  // namespace seqdiff
