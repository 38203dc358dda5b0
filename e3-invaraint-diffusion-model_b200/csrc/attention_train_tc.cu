// attention_train_tc.cu -- tensor-core version of the training attention (forward with probability dropout, and the backward) for
// the 16-bit modes; same math and interface as attention_train.cu (which stays the fp32 parity path and the reference for this one).
//
// One CTA (8 warps) per (graph, head); K, V and -- for relative_key -- a window of the distance embedding E live in shared memory
// as 16-bit tiles; queries are walked in blocks of 32 rows.  Every product is a warp-level 16x16x16 MMA (nvcuda::wmma, fp32
// accumulation) on shared-memory operands:
//     S  = Q K^T            QE = Q Ewin^T          dP = dO V^T                       (scores; relative term; upstream of the softmax)
//     dQ = dS K + dSk Ewin  dK += dS^T Q           dV += drop(P)^T dO   dEwin += dSk^T Q
// where S[l,r] += QE[l, l + 127 - r] (the relative_key skew: key r of query l sits on diagonal l - r) and dSk[l, l + 127 - r] = dS[l,r]
// is the same skew applied to the score gradient.  Softmax, dropout (Philox, regenerated -- nothing of size L x L touches HBM) and the
// dS formula run in fp32 on CUDA cores between the MMA phases.  dK / dV accumulate in register fragments across the query blocks
// (warp w owns keys 16w .. 16w+15), dE accumulates per CTA in shared memory along the diagonals and is flushed with atomics.
// These are the legacy (mma.sync-class) tensor cores: this kernel is ~4 % of the training FLOPs and sized for L <= 128; the
// GEMMs that dominate the step run on tcgen05 (gemm.cu).
#include <mma.h>

#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

namespace seqdiff {
using namespace nvcuda;

constexpr int kTcThreads = 256;
constexpr int kTcQB = 32;          // query rows per block
constexpr int kTcK = 128;          // keys per CTA (padded)
constexpr int kTcW = 160;          // window rows of E per query block: 32 + 127, padded to a multiple of 16
constexpr int kLdD = 72;           // 16-bit [rows][64] tiles
constexpr int kLdK = 136;          // 16-bit [32][128] tiles
constexpr int kLdW = 168;          // 16-bit [32][160] tile
constexpr int kLdS = 132;          // fp32 [32][128]
constexpr int kLdQE = 164;         // fp32 [32][160]

struct TcSmem {  // byte offsets (every tile 32 B aligned)
  static constexpr int kK = 0;                                   // T [128][72]
  static constexpr int kV = kK + kTcK * kLdD * 2;
  static constexpr int kQ = kV + kTcK * kLdD * 2;                // T [32][72]
  static constexpr int kdO = kQ + kTcQB * kLdD * 2;
  static constexpr int kE = kdO + kTcQB * kLdD * 2;              // T [160][72]
  static constexpr int kP = kE + kTcW * kLdD * 2;                // T [32][136]  drop(P)
  static constexpr int kdS = kP + kTcQB * kLdK * 2;              // T [32][136]
  static constexpr int kdSk = kdS + kTcQB * kLdK * 2;            // T [32][168]  skewed dS
  static constexpr int kS = kdSk + kTcQB * kLdW * 2;             // f32 [32][132] scores / staging
  static constexpr int kQE = kS + kTcQB * kLdS * 4;              // f32 [32][164]
  static constexpr int kdP = kQE + kTcQB * kLdQE * 4;            // f32 [32][132]
  static constexpr int kMask = kdP + kTcQB * kLdS * 4;           // f32 [128] additive mask (0 / -10000 / -inf)
  static constexpr int kdE = kMask + kTcK * 4;                   // f32 [256][64] (REL backward)
  static constexpr int kEnd = kdE + 256 * 64 * 4;
};
static_assert(TcSmem::kEnd <= 232448, "over the 227 KB shared-memory limit");
static_assert(TcSmem::kS % 32 == 0 && TcSmem::kQE % 32 == 0 && TcSmem::kdP % 32 == 0 && TcSmem::kdE % 32 == 0 && TcSmem::kE % 32 == 0 &&
                  TcSmem::kP % 32 == 0 && TcSmem::kdS % 32 == 0 && TcSmem::kdSk % 32 == 0,
              "wmma tiles must be 32 B aligned");

template <typename T>
__device__ __forceinline__ void tc_stage(T* dst /*[max_rows][kLdD]*/, const T* __restrict__ src, int ld, int rows, int max_rows) {
  for (int e = threadIdx.x; e < max_rows * 8; e += kTcThreads) {
    const int r = e >> 3, d8 = (e & 7) * 8;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r < rows) v = *reinterpret_cast<const uint4*>(src + static_cast<size_t>(r) * ld + d8);
    *reinterpret_cast<uint4*>(dst + r * kLdD + d8) = v;
  }
}

// C[32 x (16 * n_tiles)] = A[32 x 64] * B^T, B rows = output columns ([n][64] tiles, i.e. col_major B).  Warp w takes column tiles w, w + 8, ...
template <typename T>
__device__ __forceinline__ void mm_rows32_k64_bt(const T* sA, const T* sB, int n_tiles, float* sC, int ldc, int warp) {
  for (int n = warp; n < n_tiles; n += 8) {
    wmma::fragment<wmma::accumulator, 16, 16, 16, float> c0, c1;
    wmma::fill_fragment(c0, 0.f);
    wmma::fill_fragment(c1, 0.f);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::col_major> b;
      wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::row_major> a0, a1;
      wmma::load_matrix_sync(b, sB + n * 16 * kLdD + k * 16, kLdD);
      wmma::load_matrix_sync(a0, sA + k * 16, kLdD);
      wmma::load_matrix_sync(a1, sA + 16 * kLdD + k * 16, kLdD);
      wmma::mma_sync(c0, a0, b, c0);
      wmma::mma_sync(c1, a1, b, c1);
    }
    wmma::store_matrix_sync(sC + n * 16, c0, ldc, wmma::mem_row_major);
    wmma::store_matrix_sync(sC + 16 * ldc + n * 16, c1, ldc, wmma::mem_row_major);
  }
}

template <typename T, bool REL, bool BWD>
__global__ void __launch_bounds__(kTcThreads, 1) attention_train_tc_kernel(int heads, int Lq, int Lk, const T* __restrict__ q, int ldq,
                                                                          const T* __restrict__ k, int ldk, const T* __restrict__ v, int ldv,
                                                                          const T* __restrict__ E, int P, const float* __restrict__ key_mask,
                                                                          DropSpec dr, T* __restrict__ out, const T* __restrict__ dout,
                                                                          T* __restrict__ dq, int lddq, T* __restrict__ dk, int lddk,
                                                                          T* __restrict__ dv, int lddv, float* __restrict__ dE, int n_items) {
  pdl_wait();
  extern __shared__ __align__(128) uint8_t smraw[];
  uint8_t* sm = smraw + ((128u - (smem_u32(smraw) & 127u)) & 127u);
  // (nvcuda::wmma's load_matrix_sync lowers to state-space-less wmma.load: 17 % of the executed instructions are generic LD on
  //  shared addresses -- an address-space hint does not change that; explicit ldmatrix would)
  T* sK = reinterpret_cast<T*>(sm + TcSmem::kK);
  T* sV = reinterpret_cast<T*>(sm + TcSmem::kV);
  T* sQ = reinterpret_cast<T*>(sm + TcSmem::kQ);
  T* sdO = reinterpret_cast<T*>(sm + TcSmem::kdO);
  T* sE = reinterpret_cast<T*>(sm + TcSmem::kE);
  T* sP = reinterpret_cast<T*>(sm + TcSmem::kP);
  T* sdS = reinterpret_cast<T*>(sm + TcSmem::kdS);
  T* sdSk = reinterpret_cast<T*>(sm + TcSmem::kdSk);
  float* sS = reinterpret_cast<float*>(sm + TcSmem::kS);
  float* sQE = reinterpret_cast<float*>(sm + TcSmem::kQE);
  float* sdP = reinterpret_cast<float*>(sm + TcSmem::kdP);
  float* sMask = reinterpret_cast<float*>(sm + TcSmem::kMask);
  float* sdE = reinterpret_cast<float*>(sm + TcSmem::kdE);

  const int t = threadIdx.x, warp = t >> 5;
  const int H = heads * 64;
  // dE of the distance embedding accumulates in shared memory over ALL (graph, head) items this CTA walks and is flushed once:
  // with one item per CTA every CTA sent 16 K atomics to the same 255 x 64 addresses (25 M contended atomics per launch at B = 128).
  if (REL && BWD)
    for (int e = t; e < 256 * 64; e += kTcThreads) sdE[e] = 0.f;
  const int l = t >> 3, c = t & 7;  // elementwise phases: row l of the block, keys 16 c .. 16 c + 15
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
  const int h = item % heads, b = item / heads;
  __syncthreads();  // the previous item's epilogue is done with the staging buffers
  const T* qb = q + static_cast<size_t>(b) * Lq * ldq + h * 64;
  tc_stage<T>(sK, k + static_cast<size_t>(b) * Lk * ldk + h * 64, ldk, Lk, kTcK);
  tc_stage<T>(sV, v + static_cast<size_t>(b) * Lk * ldv + h * 64, ldv, Lk, kTcK);
  for (int r = t; r < kTcK; r += kTcThreads)
    sMask[r] = r < Lk ? (1.0f - key_mask[static_cast<size_t>(b) * Lk + r]) * -10000.0f : -INFINITY;

  // dK / dV of this warp's 16 keys: 4 column tiles each, alive across the query blocks
  wmma::fragment<wmma::accumulator, 16, 16, 16, float> accK[BWD ? 4 : 1], accV[BWD ? 4 : 1];
  if (BWD) {
#pragma unroll
    for (int n = 0; n < 4; ++n) { wmma::fill_fragment(accK[n], 0.f); wmma::fill_fragment(accV[n], 0.f); }
  }
  const size_t drop_base = (static_cast<size_t>(b) * heads + h) * Lq;

  for (int q0 = 0; q0 < Lq; q0 += kTcQB) {
    __syncthreads();  // the previous block's MMAs are done with sQ / sdO / sE / sP / sdS / sdSk
    const int rows = Lq - q0 < kTcQB ? Lq - q0 : kTcQB;
    tc_stage<T>(sQ, qb + static_cast<size_t>(q0) * ldq, ldq, rows, kTcQB);
    if (BWD) tc_stage<T>(sdO, dout + (static_cast<size_t>(b) * Lq + q0) * H + h * 64, H, rows, kTcQB);
    if (REL) {
      // window row w <-> E row j = q0 + w - 127 + P - 1;  S[l][r] uses w = l + 127 - r
      const int j0 = q0 - 127 + P - 1;
      for (int e = t; e < kTcW * 8; e += kTcThreads) {
        const int w = e >> 3, d8 = (e & 7) * 8, j = j0 + w;
        uint4 x = make_uint4(0u, 0u, 0u, 0u);
        if (j >= 0 && j < 2 * P - 1) x = *reinterpret_cast<const uint4*>(E + static_cast<size_t>(j) * 64 + d8);
        *reinterpret_cast<uint4*>(sE + w * kLdD + d8) = x;
      }
    }
    __syncthreads();
    mm_rows32_k64_bt<T>(sQ, sK, kTcK / 16, sS, kLdS, warp);             // S  = Q K^T
    if (REL) mm_rows32_k64_bt<T>(sQ, sE, kTcW / 16, sQE, kLdQE, warp);  // QE = Q Ewin^T
    if (BWD) mm_rows32_k64_bt<T>(sdO, sV, kTcK / 16, sdP, kLdS, warp);  // dP = dO V^T
    __syncthreads();

    // ---- softmax (+ dropout, + dS) in fp32: thread (l, c) owns keys 16 c .. 16 c + 15 of row l ----
    const bool live = l < rows;
    float p[16];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int r = 16 * c + i;
      float sv = sS[l * kLdS + r];
      if (REL) sv += sQE[l * kLdQE + l + 127 - r];
      sv = sv * 0.125f + sMask[r];
      p[i] = sv;
      mx = fmaxf(mx, sv);
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      p[i] = expf(p[i] - mx);  // keys >= Lk carry -inf -> 0
      sum += p[i];
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.0f / sum;
    float keep[16];
    {
      uint64_t last_q = ~0ull;
      uint32_t w4[4] = {0u, 0u, 0u, 0u};
      const uint32_t thr = dr.p > 0.f ? static_cast<uint32_t>(static_cast<double>(dr.p) * 4294967296.0) : 0u;
      const float sc = dr.p > 0.f ? 1.0f / (1.0f - dr.p) : 1.0f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int r = 16 * c + i;
        float kp = (live && r < Lk) ? 1.0f : 0.f;
        if (dr.p > 0.f && kp != 0.f) {
          const size_t e = (drop_base + q0 + l) * Lk + r;
          if ((e >> 2) != last_q) {
            last_q = e >> 2;
            w4[0] = static_cast<uint32_t>(last_q); w4[1] = static_cast<uint32_t>(last_q >> 32); w4[2] = dr.site; w4[3] = dr.step;
            philox4x32_10(w4, static_cast<uint32_t>(dr.seed), static_cast<uint32_t>(dr.seed >> 32));
          }
          kp = w4[e & 3] >= thr ? sc : 0.f;
        }
        keep[i] = kp;
        p[i] *= inv;
      }
    }
    if (BWD) {
      float dp[16], dot = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        dp[i] = sdP[l * kLdS + 16 * c + i] * keep[i];
        dot = fmaf(dp[i], p[i], dot);
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      float pd[2][8], dsv[2][8];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int r = 16 * c + i;
        const float ds = live ? p[i] * (dp[i] - dot) * 0.125f : 0.f;
        dsv[i >> 3][i & 7] = ds;
        pd[i >> 3][i & 7] = p[i] * keep[i];
        if (REL) sdSk[l * kLdW + l + 127 - r] = from_f32<T>(ds);  // skewed copy: row-dependent offset, scalar stores
      }
      // 16 consecutive keys per thread: two 128-bit stores per tile (scalar 2-byte stores were 23 % of the stall samples, 46 % of
      // the shared-memory wavefronts excess)
      store8<T>(sP + l * kLdK + 16 * c, pd[0]);
      store8<T>(sP + l * kLdK + 16 * c + 8, pd[1]);
      store8<T>(sdS + l * kLdK + 16 * c, dsv[0]);
      store8<T>(sdS + l * kLdK + 16 * c + 8, dsv[1]);
      if (REL) {  // window columns outside [l, l + 127] of row l hold no key: zeros (4 of the 32 per thread)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int z = 4 * c + i;             // 0..31
          const int w = z < l ? z : z + 128;   // [0, l) then (l + 127, 159]
          if (w < kTcW) sdSk[l * kLdW + w] = from_f32<T>(0.f);
        }
      }
    } else {
      float pd[2][8];
#pragma unroll
      for (int i = 0; i < 16; ++i) pd[i >> 3][i & 7] = p[i] * keep[i];
      store8<T>(sP + l * kLdK + 16 * c, pd[0]);
      store8<T>(sP + l * kLdK + 16 * c + 8, pd[1]);
    }
    __syncthreads();

    // ---- second-stage products ----
    {
      // [32 x 64] result: forward ctx = drop(P) V; backward dq = dS K + dSk Ewin.  Warp w: row tile w >> 2, column tile w & 3.
      const int mt = warp >> 2, nt = warp & 3;
      wmma::fragment<wmma::accumulator, 16, 16, 16, float> acc;
      wmma::fill_fragment(acc, 0.f);
      const T* A = (BWD ? sdS : sP) + mt * 16 * kLdK;
      const T* Bm = BWD ? sK : sV;
#pragma unroll
      for (int kk = 0; kk < kTcK / 16; ++kk) {
        wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::row_major> a;
        wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::row_major> bf;
        wmma::load_matrix_sync(a, A + kk * 16, kLdK);
        wmma::load_matrix_sync(bf, Bm + kk * 16 * kLdD + nt * 16, kLdD);
        wmma::mma_sync(acc, a, bf, acc);
      }
      if (REL && BWD) {
#pragma unroll
        for (int kk = 0; kk < kTcW / 16; ++kk) {
          wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::row_major> a;
          wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::row_major> bf;
          wmma::load_matrix_sync(a, sdSk + mt * 16 * kLdW + kk * 16, kLdW);
          wmma::load_matrix_sync(bf, sE + kk * 16 * kLdD + nt * 16, kLdD);
          wmma::mma_sync(acc, a, bf, acc);
        }
      }
      wmma::store_matrix_sync(sS + mt * 16 * kLdS + nt * 16, acc, kLdS, wmma::mem_row_major);  // staging (scores are consumed)
    }
    if (BWD) {
      // dK / dV of this warp's keys: A = dS^T / drop(P)^T (col_major view of the [32][128] tiles), B = Q / dO
#pragma unroll
      for (int kk = 0; kk < kTcQB / 16; ++kk) {
        wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::col_major> as, ap;
        wmma::load_matrix_sync(as, sdS + kk * 16 * kLdK + warp * 16, kLdK);
        wmma::load_matrix_sync(ap, sP + kk * 16 * kLdK + warp * 16, kLdK);
#pragma unroll
        for (int n = 0; n < 4; ++n) {
          wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::row_major> bq, bo;
          wmma::load_matrix_sync(bq, sQ + kk * 16 * kLdD + n * 16, kLdD);
          wmma::load_matrix_sync(bo, sdO + kk * 16 * kLdD + n * 16, kLdD);
          wmma::mma_sync(accK[n], as, bq, accK[n]);
          wmma::mma_sync(accV[n], ap, bo, accV[n]);
        }
      }
      if (REL) {
        // dEwin[160 x 64] += dSk^T Q, accumulated in the CTA's diagonal buffer at rows q0 + w (q0 is a multiple of 32)
        for (int tile = warp; tile < (kTcW / 16) * 4; tile += 8) {
          const int wt = tile >> 2, nt = tile & 3;
          float* cptr = sdE + static_cast<size_t>(q0 + wt * 16) * 64 + nt * 16;
          if (q0 + wt * 16 + 16 > 256) continue;  // (cannot happen for Lq <= 128: q0 <= 96, w < 160)
          wmma::fragment<wmma::accumulator, 16, 16, 16, float> ce;
          wmma::load_matrix_sync(ce, cptr, 64, wmma::mem_row_major);
#pragma unroll
          for (int kk = 0; kk < kTcQB / 16; ++kk) {
            wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::col_major> a;
            wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::row_major> bq;
            wmma::load_matrix_sync(a, sdSk + kk * 16 * kLdW + wt * 16, kLdW);
            wmma::load_matrix_sync(bq, sQ + kk * 16 * kLdD + nt * 16, kLdD);
            wmma::mma_sync(ce, a, bq, ce);
          }
          wmma::store_matrix_sync(cptr, ce, 64, wmma::mem_row_major);
        }
      }
    }
    __syncthreads();
    // staged [32 x 64] fp32 result -> global (T), 8 elements per thread
    {
      const int rr = t >> 3, d8 = (t & 7) * 8;
      if (rr < rows) {
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = sS[rr * kLdS + d8 + j];
        T* dst = BWD ? dq + (static_cast<size_t>(b) * Lq + q0 + rr) * lddq + h * 64 + d8 : out + (static_cast<size_t>(b) * Lq + q0 + rr) * H + h * 64 + d8;
        store8<T>(dst, x);
      }
    }
  }
  if (BWD) {
    __syncthreads();
    // dK, then dV: accumulator fragments -> fp32 staging [128][64] (the score buffers: 53 KB contiguous) -> global
    float* stg = sS;
    for (int which = 0; which < 2; ++which) {
#pragma unroll
      for (int n = 0; n < 4; ++n) wmma::store_matrix_sync(stg + warp * 16 * 64 + n * 16, which == 0 ? accK[n] : accV[n], 64, wmma::mem_row_major);
      __syncthreads();
      for (int e = t; e < kTcK * 8; e += kTcThreads) {
        const int r = e >> 3, d8 = (e & 7) * 8;
        if (r < Lk) {
          float x[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) x[j] = stg[r * 64 + d8 + j];
          T* dst = which == 0 ? dk + (static_cast<size_t>(b) * Lk + r) * lddk + h * 64 + d8 : dv + (static_cast<size_t>(b) * Lk + r) * lddv + h * 64 + d8;
          store8<T>(dst, x);
        }
      }
      __syncthreads();
    }
  }
  }  // item loop
  if (BWD) {
    if (REL) {
      __syncthreads();
      // diagonal a = (l - r) + 127  <->  E row a - 127 + P - 1
      for (int e = t; e < 256 * 64; e += kTcThreads) {
        const float x = sdE[e];
        const int j = (e >> 6) - 127 + P - 1;
        if (x != 0.f && j >= 0 && j < 2 * P - 1) atomicAdd(dE + static_cast<size_t>(j) * 64 + (e & 63), x);
      }
    }
  }
}

template <typename T, bool REL, bool BWD>
static int launch_tc_at(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* E, int P,
                        const float* mask, DropSpec dr, T* out, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE,
                        cudaStream_t s) {
  auto kfn = attention_train_tc_kernel<T, REL, BWD>;
  const size_t smem = static_cast<size_t>((REL && BWD) ? TcSmem::kEnd : TcSmem::kdE) + 128;
  static bool configured = false;
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::kEnd + 128));
    configured = true;
  }
  // REL backward: a few items per CTA so that the dE flush (16 K atomics per CTA) is amortised; otherwise one item per CTA
  const int n_items = B * heads;
  int grid = n_items;
  if (REL && BWD) { const int cap = 2 * num_sms(); if (grid > cap) grid = cap; }
  SD_CUDA(launch_k(kfn, dim3(grid), dim3(kTcThreads), smem, s, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, E, P, mask, dr, out, dout, dq, lddq, dk, lddk,
                   dv, lddv, dE, n_items));
  SD_LAUNCHED(BWD ? "attention_bwd_tc" : "attention_train_fwd_tc", s);
  return SEQDIFF_OK;
}

static int check_tc(int B, int heads, int Lq, int Lk, int ldq, int ldk, int ldv, const void* E, int P, int lddq, int lddk, int lddv) {
  SD_CHECK(B > 0 && heads > 0 && Lq > 0 && Lk > 0, "empty attention");
  SD_CHECK(Lk <= kTcK && Lq <= 128, "training attention: sequence length is limited to 128 (reference training uses max_seq_len 64 / 128)");
  SD_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && lddq % 8 == 0 && lddk % 8 == 0 && lddv % 8 == 0, "row strides must be multiples of 8 elements");
  SD_CHECK(!E || (Lq <= P && Lk <= P), "relative_key: sequence longer than max_position_embeddings");
  return SEQDIFF_OK;
}

template <typename T>
int attention_train_fwd_tc(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                           const float* key_mask, DropSpec dr, T* out, cudaStream_t s) {
  SD_TRY(check_tc(B, heads, Lq, Lk, ldq, ldk, ldv, dist_emb, P, 8, 8, 8));
  if (dist_emb)
    return launch_tc_at<T, true, false>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, out, nullptr, nullptr, 0, nullptr, 0, nullptr, 0,
                                        nullptr, s);
  return launch_tc_at<T, false, false>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, out, nullptr, nullptr, 0, nullptr, 0, nullptr, 0,
                                       nullptr, s);
}
template <typename T>
int attention_bwd_tc(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                     const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s) {
  SD_TRY(check_tc(B, heads, Lq, Lk, ldq, ldk, ldv, dist_emb, P, lddq, lddk, lddv));
  SD_CHECK(dout && dq && dk && dv && (!dist_emb || dE), "attention_bwd: null argument");
  if (dist_emb)
    return launch_tc_at<T, true, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, nullptr, dout, dq, lddq, dk, lddk, dv, lddv, dE, s);
  return launch_tc_at<T, false, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, nullptr, dout, dq, lddq, dk, lddk, dv, lddv, dE, s);
}
#define SD_INST_TCAT(T)                                                                                                                               \
  template int attention_train_fwd_tc<T>(int, int, int, int, const T*, int, const T*, int, const T*, int, const T*, int, const float*, DropSpec, T*, \
                                         cudaStream_t);                                                                                              \
  template int attention_bwd_tc<T>(int, int, int, int, const T*, int, const T*, int, const T*, int, const T*, int, const float*, DropSpec, const T*, \
                                   T*, int, T*, int, T*, int, float*, cudaStream_t)
SD_INST_TCAT(bf16);
SD_INST_TCAT(f16);

}  // namespace seqdiff
