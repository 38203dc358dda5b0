// attention_pipe.cu -- persistent, warp-specialised tcgen05 attention core (same math as attention.cu / attention_tc.cu,
// SURVEY.md Appendix A; reference call sites sequence_model/model.py:61 and 226-231 through HF BertSelfAttention):
//
//   S[l,r] = ( q_l . k_r + q_l . E[l - r + P - 1] ) / 8 + (1 - mask[r]) * -10000 ;  out_l = softmax_r(S[l,:]) @ V
//
// attention_tc.cu runs ONE (graph, head, query block) per CTA as a serial chain  TMA -> MMA -> softmax -> MMA -> store; at
// L = 128 that chain is pure latency (25-41 us per launch for 3-6 GFLOP).  Here one CTA per SM walks a list of work items
// (graph, head, 128-query block) x key blocks ("steps") with three roles that only meet at mbarriers:
//   warp 0      TMA producer : Q (double-buffered per item), K (+ the 256-row window of E a step can touch), V (double-buffered)
//   warp 1      MMA issuer   : S = Q K^T and QE = Q Ewin^T for step g+1 are issued as soon as the softmax threads have DRAINED
//                              S / QE of step g from TMEM into registers -- i.e. under step g's exp / P / PV work;  O (+)= P V
//   warps 2..9  softmax      : two threads per query row (TMEM lane), each owning two interleaved 32-key chunks of the step: relative-key skew
//                              by a register barrel shift, scale + mask, online softmax, P -> smem (SW128 K-major A operand),
//                              O rescale in TMEM when the running maximum moves.
// Masked keys: a 32-key chunk whose keys are all masked contributes exp2(s - 10000 log2e - m) = 0 exactly (fp32 underflow, the
// same underflow the reference's additive -10000 relies on), so its TMEM load, skew, scores and exp2 are skipped and zeros go
// into P -- bit-identical P, half the MUFU work on ragged pockets.  (Chunk 0 of an item's first step is always computed, so
// a row never ends with an empty sum; only a sequence with NO unmasked key at all deviates from the reference, which then
// attends uniformly over padding.)
// The O epilogue of an item is deferred into the first step of the next item (O is double-buffered in TMEM) and the exp2 of a
// step runs before the wait on the previous step's PV, so no role ever waits on an MMA it has just triggered.  TMEM: REL  S 128 | QE 256 | O 2x64 = 512 columns; no-REL  S 2x128 | O 2x64.
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"
#include "skew.cuh"

namespace seqdiff {

unsigned long long* g_attn_trace = nullptr;  // debug timeline buffer (4 x 1024 u64), set through seqdiff_debug_attn_trace

constexpr int kPQ = 128;            // query rows per item (= UMMA M = TMEM lanes)
constexpr int kPK = 128;            // keys per step
constexpr int kPipeThreads = 320;   // warp 0 TMA, warp 1 MMA, warps 2..9 softmax
constexpr int kSoftThreads = 256;
constexpr float kLog2e = 1.44269504088896f;

template <bool REL> struct PipeCfg {
  static constexpr int kNKS = REL ? 1 : 2;                        // K (+E) smem stages
  static constexpr int kNS = REL ? 1 : 2;                         // S accumulator stages in TMEM
  static constexpr int kQ = 0;                                    // 2 x [128][64] 16-bit, SW128
  static constexpr int kK = kQ + 2 * 16384;                       // kNKS x [128][64]
  static constexpr int kE = kK + kNKS * 16384;                    // [256][64] (REL)
  static constexpr int kNVS = REL ? 1 : 2;                        // V smem stages (REL: smem is full; PV(g) is a whole step after PV(g-1))
  static constexpr int kV = kE + (REL ? 32768 : 0);               // kNVS x [128][64]
  static constexpr int kP = kV + kNVS * 16384;                    // [2 key halves][128][64]
  static constexpr int kOut = kP + 32768;                         // [128][64] 16-bit output staging tile (16B chunks XOR-swizzled by row & 7)
  static constexpr int kMask = kOut + 16384;                      // 2 x [128] fp32 (step parity)
  static constexpr int kXch = kMask + 2 * kPK * 4;                // [step parity][key half][128] row maxima
  static constexpr int kLsum = kXch + 2 * 2 * kPQ * 4;            // [item parity][key half][128] row sums
  static constexpr int kFlag = kLsum + 2 * 2 * kPQ * 4;           // [step parity][4] int: 32-key chunk holds at least one unmasked key
  static constexpr int kBar = kFlag + 64;                         // mbarriers + tmem slot
  static constexpr int kBytes = kBar + 256 + 1024;                // + alignment slack
  static constexpr int kColS = 0;
  static constexpr int kColQE = 128;
  static constexpr int kColO = REL ? 384 : 256;
};

__device__ __forceinline__ void soft_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void soft_bar2_sync() { asm volatile("bar.sync 2, 256;" ::: "memory"); }

struct PipeItem {
  int b, h, q0;
};
__device__ __forceinline__ PipeItem decode_item(int item, int nqb, int heads) {
  PipeItem r;
  r.q0 = (item % nqb) * kPQ;
  const int bh = item / nqb;
  r.h = bh % heads;
  r.b = bh / heads;
  return r;
}
// Walks this CTA's step list (item = blockIdx.x + it * gridDim.x; kb = 0..nkb-1) without divisions in the loop: the item
// stride is decomposed once into (db, dh, dqb) and applied with carries.  (An integer division per step sat on the softmax
// threads' critical path: ~800 cycles per item in the timeline.)  KV: the key graph kg = b / kv_div is carried the same way
// (kr = b % kv_div); otherwise the key graph is b.
template <bool KV>
struct StepCursor {
  int b, h, qb, kb, it, kg_, kr;
  int db, dh, dqb, nqb, heads, nkb, dkg, dkr, kv_div;
  __device__ __forceinline__ void init(int first_item, int stride, int nqb_, int heads_, int nkb_, int kv_div_) {
    nqb = nqb_; heads = heads_; nkb = nkb_;
    const PipeItem w = decode_item(first_item, nqb, heads);
    b = w.b; h = w.h; qb = w.q0 / kPQ; kb = 0; it = 0;
    dqb = stride % nqb;
    const int sh = stride / nqb;
    dh = sh % heads;
    db = sh / heads;
    if constexpr (KV) {
      kv_div = kv_div_;
      kg_ = b / kv_div; kr = b % kv_div;
      dkg = db / kv_div; dkr = db % kv_div;
    }
  }
  __device__ __forceinline__ void next_item() {
    qb += dqb;
    if (qb >= nqb) { qb -= nqb; ++h; }
    h += dh;
    if (h >= heads) {
      h -= heads; ++b;
      if constexpr (KV) ++kr;
    }
    b += db;
    if constexpr (KV) {
      kr += dkr;
      kg_ += dkg;
      if (kr >= kv_div) { kr -= kv_div; ++kg_; }  // kr <= 2 kv_div - 1 here: one subtraction suffices
    }
    kb = 0;
    ++it;
  }
  __device__ __forceinline__ int kg() const {
    if constexpr (KV) return kg_;
    else return b;
  }
  __device__ __forceinline__ void next_step() {
    if (++kb == nkb) next_item();
  }
  __device__ __forceinline__ PipeItem item() const { return PipeItem{b, h, qb * kPQ}; }
};

// DROP: training-mode forward -- the attention-probability dropout of HF BertSelfAttention (Appendix A: A = dropout(softmax(S))) is
// applied to P just before it becomes the A operand of P V; the row sums that normalise the output use the un-dropped
// probabilities.  Mask of element e = ((b * heads + h) * Lq + l) * Lk + r: word e & 3 of Philox4x32-10(counter (e >> 2, site, step),
// key seed) -- the indexing of attention_train.cu / attention_train_tc.cu, whose backward kernels regenerate the same mask.
template <typename T, bool REL, bool DROP = false>
__global__ void __launch_bounds__(kPipeThreads, 1)
attention_pipe_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                      const __grid_constant__ CUtensorMap tmE, const __grid_constant__ CUtensorMap tmO, const float* __restrict__ key_mask, int heads, int Lq,
                      int Lk, int P, uint32_t fmt, int nqb, int n_items, unsigned long long* __restrict__ trace, const int* __restrict__ q_off,
                      const int* __restrict__ k_off, const int* __restrict__ q_len, int Lk_mask, int kv_div, T* __restrict__ out_raw,
                      const DropSpec dr, uint32_t* __restrict__ keep_out) {
  // keep_out (DROP, Lq / Lk <= 128, optional): the dropout mask of item (b, h) as bits -- word ((b * heads + h) * 128 + row) * 4 + kc holds
  // keys 32 kc .. 32 kc + 31 of query `row` -- so that the backward kernel reads 8 bytes per thread instead of regenerating 16 Philox calls
  // q_off != NULL: packed (ragged) batch -- graph b's rows start at q_off[b] / k_off[b] of the packed q / k / v matrices, Lq / Lk are
  // the largest lengths of the batch, key_mask keeps its padded pitch Lk_mask, and output rows are stored per thread with a
  // q_len[b] predicate (a bulk tile store would spill into the next graph's rows).
  // kv_div: query graph b reads the keys, values and key-mask row of graph b / kv_div (carried by the step cursors, no division
  // per step).  The training-mode kernels (DROP) always read their own graph and leave the cursor without that bookkeeping.
  using Cursor = StepCursor<!DROP>;
  using C = PipeCfg<REL>;
  constexpr int NKS = C::kNKS, NS = C::kNS, NVS = C::kNVS;
  constexpr float kScale2 = 0.125f * kLog2e;
  extern __shared__ uint8_t smem_raw[];
  // 1024B-align by OFFSET (not through an integer cast): keeps the pointer provably shared, so accesses compile to LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kBar);
  uint64_t* q_full = bars;          // [2]
  uint64_t* q_empty = bars + 2;     // [2]
  uint64_t* ke_full = bars + 4;     // [2]
  uint64_t* ke_empty = bars + 6;    // [2]
  uint64_t* v_full = bars + 8;      // [2]
  uint64_t* v_empty = bars + 10;    // [2]
  uint64_t* s_full = bars + 12;     // [2]
  uint64_t* s_empty = bars + 14;    // [2]
  uint64_t* p_full = bars + 16;
  uint64_t* o_full = bars + 17;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
  float* sMask = reinterpret_cast<float*>(smem + C::kMask);
  float* xch = reinterpret_cast<float*>(smem + C::kXch);
  float* lsum = reinterpret_cast<float*>(smem + C::kLsum);
  int* sFlag = reinterpret_cast<int*>(smem + C::kFlag);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = warp_id_uniform();  // provably warp-uniform: the TMA / MMA role loops stay on the uniform datapath
  const int nkb = (Lk + kPK - 1) / kPK;
  const int my_items = (static_cast<int>(blockIdx.x) < n_items) ? (n_items - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;

  // optional timeline (debug): CTA 0 only, one lane per role, (clock << 8 | event id) into trace[role * 1024 + n]
  int tr_n = 0;
  const bool tr_on = trace != nullptr && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 1 || warp == 2 || warp == 6);
  const int tr_base = (warp == 0 ? 0 : warp == 1 ? 1 : warp == 2 ? 2 : 3) * 1024;
  auto TR = [&](int id) {
    if (tr_on && tr_n < 1023) trace[tr_base + 1 + tr_n++] = (static_cast<unsigned long long>(clock64()) << 8) | static_cast<unsigned>(id);
  };

  if (tid == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    if (REL) tma_prefetch_desc(&tmE);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 14; ++i) mbar_init(&bars[i], 1);
    mbar_init(&s_empty[0], 8);
    mbar_init(&s_empty[1], 8);
    mbar_init(p_full, 8);
    mbar_init(o_full, 1);
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
  pdl_wait();  // key_mask / q / k / v come from the predecessor kernels

  if (warp == 0) {
    // ------------------------------------------ TMA producer ------------------------------------------
    // (whole warp runs the loop, one elected lane issues: common.cuh "warp-uniform single-issuer variants")
    {
      int g = 0;
      Cursor cur;
      cur.init(static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x), nqb, heads, nkb, kv_div);
      for (int it = 0; it < my_items; ++it, cur.next_item()) {
        const PipeItem w = cur.item();
        const int qs = it & 1;
        mbar_wait(&q_empty[qs], ((it >> 1) & 1) ^ 1);
        mbar_expect_tx_e(&q_full[qs], 16384);
        const int q_row0 = q_off ? __ldg(q_off + w.b) : w.b * Lq;
        const int k_row0 = q_off ? __ldg(k_off + cur.kg()) : cur.kg() * Lk;
        tma_load_2d_e(smem + C::kQ + qs * 16384, &tmQ, &q_full[qs], w.h * 64, q_row0 + w.q0);
        for (int kb = 0; kb < nkb; ++kb, ++g) {
          const int ks = g % NKS;
          mbar_wait(&ke_empty[ks], ((g / NKS) & 1) ^ 1);
          TR(1);
          mbar_expect_tx_e(&ke_full[ks], REL ? 16384 + 32768 : 16384);
          tma_load_2d_e(smem + C::kK + ks * 16384, &tmK, &ke_full[ks], w.h * 64, k_row0 + kb * kPK);
          if (REL) tma_load_2d_e(smem + C::kE, &tmE, &ke_full[ks], 0, w.q0 - kb * kPK + P - 1 - 127);
          const int vs = g % NVS;
          mbar_wait(&v_empty[vs], ((g / NVS) & 1) ^ 1);
          TR(2);
          mbar_expect_tx_e(&v_full[vs], 16384);
          tma_load_2d_e(smem + C::kV + vs * 16384, &tmV, &v_full[vs], w.h * 64, k_row0 + kb * kPK);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------ MMA issuer --------------------------------------------
    {
      const uint32_t idesc_s = umma_idesc_16(kPQ, 128, fmt, fmt);
      const uint32_t idesc_e = umma_idesc_16(kPQ, 256, fmt, fmt);
      const uint32_t idesc_o = umma_idesc_16(kPQ, 64, fmt, fmt) | (1u << 16);  // B (= V) is MN-major
      const int G = my_items * nkb;
      auto issue_s = [&](int g, int it, int kb) {
        const int qs = it & 1, ks = g % NKS, ss = g % NS;
        if (kb == 0) mbar_wait(&q_full[qs], (it >> 1) & 1);
        mbar_wait(&ke_full[ks], (g / NKS) & 1);
        TR(10);
        mbar_wait(&s_empty[ss], ((g / NS) & 1) ^ 1);  // softmax threads have drained this S (+QE) stage
        tc_fence_after();
        TR(11);
        const uint32_t qa = smem_u32(smem + C::kQ + qs * 16384), ka = smem_u32(smem + C::kK + ks * 16384);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_e(tmem_base + C::kColS + ss * 128, umma_desc_kmajor_sw128(qa + k * 32), umma_desc_kmajor_sw128(ka + k * 32), idesc_s, k ? 1u : 0u);
        if (REL) {
          const uint32_t ea = smem_u32(smem + C::kE);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_e(tmem_base + C::kColQE, umma_desc_kmajor_sw128(qa + k * 32), umma_desc_kmajor_sw128(ea + k * 32), idesc_e, k ? 1u : 0u);
        }
        umma_commit_e(&s_full[ss]);
        umma_commit_e(&ke_empty[ks]);
        if (kb == nkb - 1) umma_commit_e(&q_empty[qs]);
        TR(12);
      };
      if (G > 0) issue_s(0, 0, 0);
      int it = 0, kb = 0;        // (item, key block) of step g
      int it_s = 0, kb_s = 0;    // ... of step g + 1
      for (int g = 0; g < G; ++g) {
        if (++kb_s == nkb) { kb_s = 0; ++it_s; }
        if (g + 1 < G) issue_s(g + 1, it_s, kb_s);
        mbar_wait(p_full, g & 1);
        TR(13);
        mbar_wait(&v_full[g % NVS], (g / NVS) & 1);
        tc_fence_after();
        TR(14);
        const uint32_t pa = smem_u32(smem + C::kP), va = smem_u32(smem + C::kV + (g % NVS) * 16384);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          umma_bf16_e(tmem_base + C::kColO + (it & 1) * 64, umma_desc_kmajor_sw128(pa + (k >> 2) * 16384 + (k & 3) * 32),
                    umma_desc_kmajor_sw128(va + k * 2048), idesc_o, (kb | k) ? 1u : 0u);
        umma_commit_e(o_full);
        umma_commit_e(&v_empty[g % NVS]);
        TR(15);
        if (++kb == nkb) { kb = 0; ++it; }
      }
    }
  } else {
    // ------------------------------------------ softmax threads ---------------------------------------
    const int st = tid - 64;          // 0..255
    const int wq = warp & 3;          // TMEM lane quarter this warp may access
    const int hf = (warp - 2) >> 2;   // which 64-key half of a step this thread owns
    const int row = wq * 32 + lane;   // query row inside the item = TMEM lane
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(wq * 32) << 16);
    // additive key mask (log2 domain) of a step: fetched from global TWO steps ahead (raw value parked in a register across a
    // whole step, so its latency never shows), stored to smem one step ahead, published by that step's barrier
    auto mask_cvt = [&](float raw, bool in_range) -> float { return in_range ? (1.0f - raw) * (-10000.0f * kLog2e) : -INFINITY; };
    // raw mask value of key 128 kb + st for the step the cursor points at (false past the end of the list / for st >= 128)
    auto mask_fetch = [&](const Cursor& c, float& raw, bool& in_range) -> bool {
      if (c.it >= my_items || st >= kPK) return false;
      const int r = c.kb * kPK + st;
      in_range = r < Lk_mask;
      raw = in_range ? __ldg(key_mask + static_cast<size_t>(c.kg()) * Lk_mask + r) : 0.f;
      return true;
    };
    // O of a finished item -> global.  Each thread scales its 32 of the row's 64 output columns and drops them as 16-bit into
    // the SW128 staging tile; after a barrier one thread hands the tile to a TMA store (direct per-row stores: 32 partial
    // lines per warp instruction, ~1000 LSU cycles per item).  The tile is reused one item later: thread 0 waits for the
    // store to have read it (tma_store_wait_read) before the barrier that precedes the next epilogue.
    auto epilogue = [&](const PipeItem& w, int pit) {
      const float inv = 1.0f / (lsum[((pit & 1) * 2 + 0) * kPQ + row] + lsum[((pit & 1) * 2 + 1) * kPQ + row]);
      uint32_t r[32];
      tmem_ld_32x32(t_lane + C::kColO + (pit & 1) * 64 + hf * 32, r);
      tmem_ld_wait();
      if (q_off) {  // packed batch: 64 B per thread straight to its own row, rows past the graph's length are not written
        if (w.q0 + row < __ldg(q_len + w.b)) {
          T* dst = out_raw + (static_cast<size_t>(__ldg(q_off + w.b)) + w.q0 + row) * (static_cast<size_t>(heads) * 64) + w.h * 64 + hf * 32;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 v;
            v.x = pack2<T>(__uint_as_float(r[8 * j + 0]) * inv, __uint_as_float(r[8 * j + 1]) * inv);
            v.y = pack2<T>(__uint_as_float(r[8 * j + 2]) * inv, __uint_as_float(r[8 * j + 3]) * inv);
            v.z = pack2<T>(__uint_as_float(r[8 * j + 4]) * inv, __uint_as_float(r[8 * j + 5]) * inv);
            v.w = pack2<T>(__uint_as_float(r[8 * j + 6]) * inv, __uint_as_float(r[8 * j + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + 8 * j) = v;
          }
        }
        return;
      }
      uint8_t* orow = smem + C::kOut + row * 128;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 v;
        v.x = pack2<T>(__uint_as_float(r[8 * j + 0]) * inv, __uint_as_float(r[8 * j + 1]) * inv);
        v.y = pack2<T>(__uint_as_float(r[8 * j + 2]) * inv, __uint_as_float(r[8 * j + 3]) * inv);
        v.z = pack2<T>(__uint_as_float(r[8 * j + 4]) * inv, __uint_as_float(r[8 * j + 5]) * inv);
        v.w = pack2<T>(__uint_as_float(r[8 * j + 6]) * inv, __uint_as_float(r[8 * j + 7]) * inv);
        *reinterpret_cast<uint4*>(orow + (((hf * 4 + j) ^ (row & 7)) << 4)) = v;
      }
      fence_proxy_async_smem();  // staging writes -> visible to the TMA store (async proxy)
      soft_bar2_sync();
      if (st == 0) {  // one 16 KB bulk store per item; rows >= Lq of the graph are clipped by the [B][Lq][H] tensor map
        tma_store_3d(&tmO, smem + C::kOut, w.h * 64, w.q0, w.b);
        tma_store_commit();
      }
    };

    // mask value of key 128 kb + st of a step -> smem; warps 2..5 (st < 128) own one 32-key chunk each and record whether the
    // chunk holds any unmasked key (warp-uniform call sites only)
    auto mask_store = [&](int parity, float v, bool first_step_of_item) {
      sMask[parity * kPK + st] = v;
      const unsigned any = __ballot_sync(0xffffffffu, v == 0.0f);
      if (lane == 0) sFlag[parity * 4 + (st >> 5)] = (any != 0u || (first_step_of_item && st < 32)) ? 1 : 0;
    };
    PipeItem prev{0, 0, 0};
    Cursor cur, ahead;  // current step / the step two ahead (mask prefetch)
    cur.init(static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x), nqb, heads, nkb, kv_div);
    ahead = cur;
    if (my_items > 0) {
      float raw; bool inr;
      if (mask_fetch(ahead, raw, inr)) mask_store(0, mask_cvt(raw, inr), ahead.kb == 0);
      ahead.next_step();
      if (mask_fetch(ahead, raw, inr)) mask_store(1, mask_cvt(raw, inr), ahead.kb == 0);
      ahead.next_step();
    }
    soft_bar_sync();
    int g = 0;
    float m_raw = 0.f;
    bool m_inr = false, m_have = false, m_first = false;
    for (int it = 0; it < my_items; ++it, cur.next_item()) {
      const PipeItem w = cur.item();
      SD_DEV_ASSERT(w.b >= 0 && w.h >= 0 && w.h < heads && (w.b * heads + w.h) * nqb + w.q0 / kPQ < n_items);  // the division-free cursor stays on the item list
      SD_DEV_ASSERT(cur.kg() == w.b / kv_div);  // ... and on the key graph
      SD_DEV_ASSERT(!q_off || (__ldg(q_len + w.b) > 0 && __ldg(q_len + w.b) <= Lq && __ldg(q_off + w.b) >= 0));
      float m_run = -INFINITY, l_run = 0.f;
      for (int kb = 0; kb < nkb; ++kb, ++g) {
        const int ss = g % NS;
        TR(20);
        mbar_wait(&s_full[ss], (g / NS) & 1);
        tc_fence_after();
        TR(21);
        // ---- scores of (row, key half): S + skewed QE, scaled, masked (log2 domain) ----
        float t[2][32];
        // the two threads of a row own INTERLEAVED 32-key chunks (thread hf: chunks hf and hf + 2), so that a prefix mask --
        // peptides of 5..64 residues in 128 slots -- leaves both threads with the same number of live chunks
        const bool cv0 = sFlag[(g & 1) * 4 + hf] != 0, cv1 = sFlag[(g & 1) * 4 + hf + 2] != 0;  // warp-uniform
        const float* mk = sMask + (g & 1) * kPK + 32 * hf;  // chunk c of this thread: + 64 c
        float mx = -INFINITY;
        // (static dispatch on the chunk flags: a run-time condition around the register arrays sends them to local memory)
        auto score_chunk = [&](auto c_tag) {
          constexpr int c = decltype(c_tag)::value;
          uint32_t x0[32], x1[32];  // X[k] = k < 32 ? x0[k] : x1[k - 32]  (two arrays: no address arithmetic across them, stays in registers)
          if (REL) {
            // relative-key skew in registers.  Keys r of chunk kc = hf + 2c pair with window columns j = row + 127 - r; for
            // the warp's 32 rows that is the 2-chunk band of QE starting at chunk qc0 = wq - kc + 3 (warp-uniform), and with
            // X = those 64 columns of this lane's row:  QE[row, j(r)] = X[lane + 31 - (r - 32 kc)].  The lane-dependent
            // offset is applied by a 5-stage barrel shift (186 selects on the ALUs of all four sub-partitions); the earlier
            // scatter through a private smem row was bound by the SM's single LSU: 2.6 k cycles per item.
            const int qc0 = wq - (hf + 2 * c) + 3;
            tmem_ld_32x32(t_lane + C::kColQE + qc0 * 32, x0);
            tmem_ld_32x32(t_lane + C::kColQE + (qc0 + 1) * 32, x1);
            tmem_ld_wait();
            const uint32_t ul = static_cast<uint32_t>(lane);
            shift_stage<16>(x0, x1, ul & 16u);
            shift_stage<8>(x0, x1, ul & 8u);
            shift_stage<4>(x0, x1, ul & 4u);
            shift_stage<2>(x0, x1, ul & 2u);
            shift_stage<1>(x0, x1, ul & 1u);
          }
          uint32_t r[32];
          tmem_ld_32x32(t_lane + C::kColS + ss * 128 + (hf + 2 * c) * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float sv = __uint_as_float(r[j]);
            if (REL) sv += __uint_as_float(x0[31 - j]);
            sv = fmaf(sv, kScale2, mk[c * 64 + j]);
            t[c][j] = sv;
            mx = fmaxf(mx, sv);
          }
        };
        if (cv0 && cv1) {
          score_chunk(std::integral_constant<int, 0>{});
          score_chunk(std::integral_constant<int, 1>{});
        } else if (cv0) {
          score_chunk(std::integral_constant<int, 0>{});
        } else if (cv1) {
          score_chunk(std::integral_constant<int, 1>{});
        }
        // S (+QE) of this step now live in registers: hand the TMEM stage back so the MMAs of step g+1 run under the rest
        TR(22);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_empty[ss]);
        xch[((g & 1) * 2 + hf) * kPQ + row] = mx;
        if (g > 0 && m_have) mask_store((g + 1) & 1, mask_cvt(m_raw, m_inr), m_first);  // step g+1's mask (fetched during step g-1)
        TR(23);
        if (st == 0) tma_store_wait_read();  // previous item's output tile has left smem (next epilogue may overwrite it)
        soft_bar_sync();
        TR(24);
        m_have = mask_fetch(ahead, m_raw, m_inr);  // step g + 2
        m_first = ahead.kb == 0;
        ahead.next_step();
        const float m_new = fmaxf(m_run, fmaxf(mx, xch[((g & 1) * 2 + (hf ^ 1)) * kPQ + row]));
        const float corr = (m_run == -INFINITY) ? 0.f : ex2_approx(m_run - m_new);
        m_run = m_new;

        // ---- p = exp2(t - m) in place (MUFU-bound: runs under the PV of the previous step) ----
        float rs = 0.f;
        auto exp_chunk = [&](auto c_tag) {
          constexpr int c = decltype(c_tag)::value;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            t[c][j] = ex2_approx(t[c][j] - m_new);
            rs += t[c][j];
          }
        };
        auto zero_chunk = [&](auto c_tag) {  // every key of the chunk is masked: its probabilities underflow to exactly 0
          constexpr int c = decltype(c_tag)::value;
#pragma unroll
          for (int j = 0; j < 32; ++j) t[c][j] = 0.f;
        };
        if (cv0 && cv1) {
          exp_chunk(std::integral_constant<int, 0>{});
          exp_chunk(std::integral_constant<int, 1>{});
        } else if (cv0) {
          exp_chunk(std::integral_constant<int, 0>{});
          zero_chunk(std::integral_constant<int, 1>{});
        } else if (cv1) {
          zero_chunk(std::integral_constant<int, 0>{});
          exp_chunk(std::integral_constant<int, 1>{});
        } else {
          zero_chunk(std::integral_constant<int, 0>{});
          zero_chunk(std::integral_constant<int, 1>{});
        }
        l_run = l_run * corr + rs;
        if (kb == nkb - 1) lsum[((it & 1) * 2 + hf) * kPQ + row] = l_run;
        if (DROP) {
          // keys of chunk c: r = 128 kb + 64 c + 32 hf + j; one Philox call serves 4 consecutive keys (Lk % 4 == 0: groups never
          // straddle a row).  Fully masked chunks hold exact zeros already.
          const uint32_t thr = static_cast<uint32_t>(static_cast<double>(dr.p) * 4294967296.0);
          const float sc = 1.0f / (1.0f - dr.p);
          const size_t e_row = ((static_cast<size_t>(w.b) * heads + w.h) * Lq + w.q0 + row) * Lk + kb * kPK + 32 * hf;
          auto drop_chunk = [&](auto c_tag) {
            constexpr int c = decltype(c_tag)::value;
            uint32_t bits = 0u;
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const uint64_t qd = (e_row + 64 * c + 4 * j4) >> 2;
              uint32_t w4[4] = {static_cast<uint32_t>(qd), static_cast<uint32_t>(qd >> 32), dr.site, dr.step};
              philox4x32_10(w4, static_cast<uint32_t>(dr.seed), static_cast<uint32_t>(dr.seed >> 32));
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const bool kp = w4[u] >= thr;
                t[c][4 * j4 + u] *= (kp ? sc : 0.f);
                bits |= (kp ? 1u : 0u) << (4 * j4 + u);
              }
            }
            if (keep_out) keep_out[((static_cast<size_t>(w.b) * heads + w.h) * 128 + row) * 4 + (hf + 2 * c)] = bits;
          };
          if (cv0) drop_chunk(std::integral_constant<int, 0>{});
          if (cv1) drop_chunk(std::integral_constant<int, 1>{});
        }

        // PV of the previous step complete: the P tile is free again and O of this item may be rescaled
        if (g > 0) {
          mbar_wait(o_full, (g - 1) & 1);
          tc_fence_after();
        }
        TR(25);
        if (kb > 0 && __any_sync(0xffffffffu, corr != 1.0f)) {
          uint32_t r[32];
          tmem_ld_32x32(t_lane + C::kColO + (it & 1) * 64 + hf * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * corr);
          tmem_st_32x32(t_lane + C::kColO + (it & 1) * 64 + hf * 32, r);
          tmem_st_wait();
        }
        TR(26);
        // ---- P -> smem (A operand, K-major; SW128 tile c holds keys 64 c .. 64 c + 63): this thread's chunk c = keys
        //      64 c + 32 hf .. + 31 = 16 B chunks 4 hf .. 4 hf + 3 of the row in tile c ----
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint8_t* prow16 = smem + C::kP + c * 16384 + row * 128;
#pragma unroll
          for (int qd = 0; qd < 4; ++qd) {
            const float* p = &t[c][qd * 8];
            *reinterpret_cast<uint4*>(prow16 + (((hf * 4 + qd) ^ (row & 7)) << 4)) =
                make_uint4(pack2<T>(p[0], p[1]), pack2<T>(p[2], p[3]), pack2<T>(p[4], p[5]), pack2<T>(p[6], p[7]));
          }
        }
        fence_proxy_async_smem();  // generic-proxy smem writes (P) -> visible to the tensor core (async proxy)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
        TR(27);
        // O of the previous item (other O buffer; complete since the o_full wait above) leaves under this step's PV
        if (kb == 0 && it > 0) epilogue(prev, it - 1);
        TR(28);
      }
      prev = w;
    }
    if (my_items > 0) {
      if (st == 0) tma_store_wait_read();  // the staging tile of the item before last has left smem
      soft_bar_sync();  // publishes the last item's row sums
      mbar_wait(o_full, (g - 1) & 1);
      tc_fence_after();
      epilogue(prev, my_items - 1);
      if (st == 0) tma_store_wait_all();
    }
  }

  if (tr_on) trace[tr_base] = static_cast<unsigned long long>(tr_n);
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <typename T> struct PipeFmt;
template <> struct PipeFmt<f16> { static constexpr int v = 0; };
template <> struct PipeFmt<bf16> { static constexpr int v = 1; };

template <typename T, bool REL, bool DROP = false>
static int launch_pipe(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* E, int P,
                       const float* mask, T* out, cudaStream_t s, const AttnPack* pk, const DropSpec dr = DropSpec{0.f, 0u, 0u, 0ull},
                       uint32_t* keep_out = nullptr, int kv_div = 1) {
  using C = PipeCfg<REL>;
  auto kfn = attention_pipe_kernel<T, REL, DROP>;
  static bool configured = false;
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kBytes));
    configured = true;
  }
  constexpr int fmt = PipeFmt<T>::v;
  CUtensorMap tq, tk, tv, te, to;
  SD_TRY(make_tmap(q, fmt, pk ? pk->q_rows : B * Lq, ldq, 128, &tq));
  if (pk) to = tq;  // packed: per-thread predicated stores, no tile store
  else SD_TRY(make_tmap_3d(out, fmt, B, Lq, heads * 64, 128, &to));
  SD_TRY(make_tmap(k, fmt, pk ? pk->k_rows : B / kv_div * Lk, ldk, 128, &tk));
  SD_TRY(make_tmap(v, fmt, pk ? pk->k_rows : B / kv_div * Lk, ldv, 128, &tv));
  if (REL) SD_TRY(make_tmap(E, fmt, 2 * P - 1, 64, 256, &te));
  else te = tq;
  const int nqb = ceil_div(Lq, kPQ);
  const int n_items = B * heads * nqb;
  // SEQDIFF_ATTN_GRID caps the grid (tests: many items per CTA on a small problem)
  static const int grid_cap = [] { const char* e = getenv("SEQDIFF_ATTN_GRID"); return e ? atoi(e) : 0; }();
  int grid = n_items < num_sms() ? n_items : num_sms();
  if (grid_cap > 0 && grid > grid_cap) grid = grid_cap;
  SD_CUDA(launch_k(kfn, dim3(grid), dim3(kPipeThreads), C::kBytes, s, tq, tk, tv, te, to, mask, heads, Lq, Lk, P, static_cast<uint32_t>(fmt), nqb,
                   n_items, g_attn_trace, pk ? pk->q_off : nullptr, pk ? pk->k_off : nullptr, pk ? pk->q_len : nullptr, pk ? pk->Lk_mask : Lk, kv_div, out, dr, keep_out));
  SD_LAUNCHED(DROP ? (REL ? "attention_pipe_rel_drop" : "attention_pipe_norel_drop") : (REL ? "attention_pipe_rel" : "attention_pipe_norel"), s);
  return SEQDIFF_OK;
}

template <typename T>
int attention_pipe(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                   const float* key_mask, T* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
  SD_CHECK(B > 0 && heads > 0 && Lq > 0 && Lk > 0, "empty attention");
  SD_CHECK(kv_div >= 1 && B % kv_div == 0, "every key graph must serve kv_div whole query graphs");
  SD_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0, "row strides must be multiples of 8 elements");
  SD_CHECK((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) % 16 == 0, "q/k/v must be 16B aligned");
  SD_CHECK(!dist_emb || (Lq <= P && Lk <= P), "sequence longer than max_position_embeddings");
  SD_CHECK(!pack || (pack->q_off && pack->k_off && pack->q_len && pack->Lk_mask >= Lk && pack->q_rows > 0 && pack->k_rows > 0), "bad packed-attention descriptor");
  const DropSpec none{0.f, 0u, 0u, 0ull};
  if (dist_emb) return launch_pipe<T, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, none, nullptr, kv_div);
  return launch_pipe<T, false>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, none, nullptr, kv_div);
}
// training-mode forward (attention-probability dropout inside the kernel); needs Lk % 4 == 0
template <typename T>
int attention_pipe_dropout(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                           const float* key_mask, DropSpec dr, T* out, cudaStream_t s, uint32_t* keep_out) {
  SD_CHECK(B > 0 && heads > 0 && Lq > 0 && Lk > 0, "empty attention");
  SD_CHECK(!keep_out || (Lq <= 128 && Lk <= 128), "the keep-bit buffer covers one 128 x 128 tile per (graph, head)");
  SD_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0, "row strides must be multiples of 8 elements");
  SD_CHECK((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) % 16 == 0, "q/k/v must be 16B aligned");
  SD_CHECK(!dist_emb || (Lq <= P && Lk <= P), "sequence longer than max_position_embeddings");
  SD_CHECK(Lk % 4 == 0, "dropout in the pipelined kernel: Lk must be a multiple of 4 (one Philox call per 4 keys of a row)");
  SD_CHECK(dr.p > 0.f && dr.p < 1.f, "dropout probability must be in (0, 1)");
  if (dist_emb) return launch_pipe<T, true, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, nullptr, dr, keep_out);
  return launch_pipe<T, false, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, nullptr, dr, keep_out);
}
template int attention_pipe_dropout<bf16>(int, int, int, int, const bf16*, int, const bf16*, int, const bf16*, int, const bf16*, int, const float*, DropSpec, bf16*, cudaStream_t, uint32_t*);
template int attention_pipe_dropout<f16>(int, int, int, int, const f16*, int, const f16*, int, const f16*, int, const f16*, int, const float*, DropSpec, f16*, cudaStream_t, uint32_t*);
template int attention_pipe<bf16>(int, int, int, int, const bf16*, int, const bf16*, int, const bf16*, int, const bf16*, int, const float*, bf16*, cudaStream_t, const AttnPack*, int);
template int attention_pipe<f16>(int, int, int, int, const f16*, int, const f16*, int, const f16*, int, const f16*, int, const float*, f16*, cudaStream_t, const AttnPack*, int);

}  // namespace seqdiff
