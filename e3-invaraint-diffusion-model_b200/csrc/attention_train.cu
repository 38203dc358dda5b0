// attention_train.cu -- attention for the TRAINING step: forward with attention-probability dropout, and the backward of the
// attention core of HF BertSelfAttention with 4.38.2 `relative_key` semantics (SURVEY.md Appendix A):
//
//   S[l,r] = (q_l . k_r + q_l . E[l - r + P - 1]) / 8 + (1 - mask[r]) * -10000 ;  P = softmax_r(S) ;  ctx_l = sum_r drop(P)[l,r] v_r
//
//   dV_r = sum_l drop(P)[l,r] dctx_l                 dP[l,r] = keep[l,r] * (dctx_l . v_r)
//   dS   = P * (dP - sum_r dP * P) / 8               dq_l = sum_r dS[l,r] (k_r + E[l - r + P - 1])
//   dk_r = sum_l dS[l,r] q_l                         dE[j] = sum over (b, h, l - r + P - 1 = j) dS[l,r] q_l
//
// One CTA per (graph, head): K and V of the head are staged in shared memory as fp32 once, queries are walked in blocks of 16
// rows; probabilities are recomputed in the backward from the stored 16-bit q, k (nothing of size L x L is ever written to HBM),
// the dropout mask is regenerated from Philox.  dE is accumulated per CTA in shared memory along the diagonals l - r and flushed
// with one atomicAdd per (diagonal, feature).  All arithmetic is fp32 SIMT (this is also the fp32 parity path); key length is
// limited to 128 (the training configurations of the reference use max_seq_len 64 / 128: train_model.py:16,21).
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

namespace seqdiff {

constexpr int kAtThreads = 256;
constexpr int kAtQB = 16;     // query rows per block
constexpr int kAtMaxK = 128;  // keys staged per CTA
constexpr int kAtD = 64;
constexpr int kAtPad = kAtD + 1;

struct AtSmem {
  // float offsets
  static constexpr int kK = 0;
  static constexpr int kV = kK + kAtMaxK * kAtPad;
  static constexpr int kQ = kV + kAtMaxK * kAtPad;
  static constexpr int kdO = kQ + kAtQB * kAtPad;
  static constexpr int kS = kdO + kAtQB * kAtPad;
  static constexpr int kdS = kS + kAtQB * (kAtMaxK + 1);
  static constexpr int kM = kdS + kAtQB * (kAtMaxK + 1);
  static constexpr int kE = kM + kAtMaxK;                         // [kAtQB + kAtMaxK - 1][kAtPad] window of E (REL)
  static constexpr int kdE = kE + (kAtQB + kAtMaxK - 1) * kAtPad;  // [2 * kAtMaxK - 1][kAtD] (REL, backward)
  static constexpr int kEnd = kdE + (2 * kAtMaxK - 1) * kAtD;
};

// scores + softmax of one block of 16 query rows.  Thread t: row l = t >> 4, keys r = (t & 15) + 16 i.  Leaves p[i] = P[l][r_i]
// (normalised, 0 for r >= Lk) in registers.
template <bool REL>
__device__ __forceinline__ void block_probs(const float* sm, int l, int c, int Lk, float (&p)[8]) {
  const float* sQ = sm + AtSmem::kQ + l * kAtPad;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int d = 0; d < kAtD; ++d) {
    const float q = sQ[d];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = c + 16 * i;
      float kv = sm[AtSmem::kK + r * kAtPad + d];
      if (REL) kv += sm[AtSmem::kE + (l + Lk - 1 - r + (r < Lk ? 0 : r - Lk + 1)) * kAtPad + d];  // clamp the window index of dead keys
      acc[i] = fmaf(q, kv, acc[i]);
    }
  }
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = c + 16 * i;
    acc[i] = r < Lk ? acc[i] * 0.125f + (1.0f - sm[AtSmem::kM + r]) * -10000.0f : -INFINITY;
    mx = fmaxf(mx, acc[i]);
  }
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    p[i] = (c + 16 * i) < Lk ? expf(acc[i] - mx) : 0.f;
    sum += p[i];
  }
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float inv = 1.0f / sum;
#pragma unroll
  for (int i = 0; i < 8; ++i) p[i] *= inv;
}

template <typename T>
__device__ __forceinline__ void stage_rows(float* dst, const T* __restrict__ src, int ld, int rows, int max_rows) {
  // dst [max_rows][kAtPad] <- src rows (64 features each); rows past `rows` are zero-filled
  for (int e = threadIdx.x; e < max_rows * (kAtD / 8); e += kAtThreads) {
    const int r = e >> 3, d8 = (e & 7) * 8;
    float v[8];
    if (r < rows) {
      load8<T>(src + static_cast<size_t>(r) * ld + d8, v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[r * kAtPad + d8 + j] = v[j];
  }
}

template <typename T, bool REL, bool BWD>
__global__ void __launch_bounds__(kAtThreads) attention_train_kernel(int heads, int Lq, int Lk, const T* __restrict__ q, int ldq,
                                                                     const T* __restrict__ k, int ldk, const T* __restrict__ v, int ldv,
                                                                     const T* __restrict__ E, int P, const float* __restrict__ key_mask,
                                                                     DropSpec dr, T* __restrict__ out, const T* __restrict__ dout,
                                                                     T* __restrict__ dq, int lddq, T* __restrict__ dk, int lddk,
                                                                     T* __restrict__ dv, int lddv, float* __restrict__ dE) {
  pdl_wait();
  extern __shared__ float sm[];
  const int h = blockIdx.x, b = blockIdx.y;
  const int t = threadIdx.x;
  const int H = heads * kAtD;
  const T* qb = q + static_cast<size_t>(b) * Lq * ldq + h * kAtD;
  const T* kb = k + static_cast<size_t>(b) * Lk * ldk + h * kAtD;
  const T* vb = v + static_cast<size_t>(b) * Lk * ldv + h * kAtD;
  stage_rows<T>(sm + AtSmem::kK, kb, ldk, Lk, kAtMaxK);
  stage_rows<T>(sm + AtSmem::kV, vb, ldv, Lk, kAtMaxK);
  for (int r = t; r < kAtMaxK; r += kAtThreads) sm[AtSmem::kM + r] = r < Lk ? key_mask[static_cast<size_t>(b) * Lk + r] : 0.f;
  if (REL && BWD)
    for (int e = t; e < (2 * kAtMaxK - 1) * kAtD; e += kAtThreads) sm[AtSmem::kdE + e] = 0.f;
  float dkr[BWD ? 32 : 1], dvr[BWD ? 32 : 1];
  if (BWD) {
#pragma unroll
    for (int d = 0; d < 32; ++d) { dkr[d] = 0.f; dvr[d] = 0.f; }
  }
  const int l = t >> 4, c = t & 15;
  const size_t drop_base = (static_cast<size_t>(b) * heads + h) * Lq;
  for (int q0 = 0; q0 < Lq; q0 += kAtQB) {
    __syncthreads();  // previous block's consumers are done with sQ / sdO / sS / sdS / sE
    const int rows = Lq - q0 < kAtQB ? Lq - q0 : kAtQB;
    stage_rows<T>(sm + AtSmem::kQ, qb + static_cast<size_t>(q0) * ldq, ldq, rows, kAtQB);
    if (BWD) stage_rows<T>(sm + AtSmem::kdO, dout + (static_cast<size_t>(b) * Lq + q0) * H + h * kAtD, H, rows, kAtQB);
    if (REL) {
      // window row w holds E[(q0 + w - (Lk - 1)) + P - 1]: S[l][r] uses w = l_loc + Lk - 1 - r
      const int j0 = q0 - (Lk - 1) + P - 1;
      for (int e = t; e < (kAtQB + Lk - 1) * (kAtD / 8); e += kAtThreads) {
        const int w = e >> 3, d8 = (e & 7) * 8;
        const int j = j0 + w;
        float x[8];
        if (j >= 0 && j < 2 * P - 1) {
          load8<T>(E + static_cast<size_t>(j) * kAtD + d8, x);
        } else {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) x[jj] = 0.f;
        }
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) sm[AtSmem::kE + w * kAtPad + d8 + jj] = x[jj];
      }
    }
    __syncthreads();
    float p[8];
    block_probs<REL>(sm, l, c, Lk, p);
    const bool live = l < rows;
    float keep[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = c + 16 * i;
      keep[i] = (live && r < Lk) ? drop_scale1(dr, (drop_base + q0 + l) * Lk + r) : 0.f;
    }
    if (BWD) {
      // dP[l][r] = keep * (dO_l . v_r);  dS = P * (dP - sum_r dP P) / 8
      float dp[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) dp[i] = 0.f;
      const float* sdO = sm + AtSmem::kdO + l * kAtPad;
      for (int d = 0; d < kAtD; ++d) {
        const float g = sdO[d];
#pragma unroll
        for (int i = 0; i < 8; ++i) dp[i] = fmaf(g, sm[AtSmem::kV + (c + 16 * i) * kAtPad + d], dp[i]);
      }
      float dot = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dp[i] *= keep[i];
        dot = fmaf(dp[i], p[i], dot);
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = c + 16 * i;
        sm[AtSmem::kdS + l * (kAtMaxK + 1) + r] = live ? p[i] * (dp[i] - dot) * 0.125f : 0.f;
        sm[AtSmem::kS + l * (kAtMaxK + 1) + r] = p[i] * keep[i];  // drop(P)
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) sm[AtSmem::kS + l * (kAtMaxK + 1) + c + 16 * i] = p[i] * keep[i];
    }
    __syncthreads();
    {
      // 16 x 64 outputs, 4 per thread: forward ctx = drop(P) V; backward dq = dS (K + E_window)
      const int d4 = c * 4;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      const float* wrow = sm + (BWD ? AtSmem::kdS : AtSmem::kS) + l * (kAtMaxK + 1);
      const float* mat = sm + (BWD ? AtSmem::kK : AtSmem::kV);
      for (int r = 0; r < Lk; ++r) {
        const float w = wrow[r];
        const float* mr = mat + r * kAtPad + d4;
        float m0 = mr[0], m1 = mr[1], m2 = mr[2], m3 = mr[3];
        if (REL && BWD) {
          const float* er = sm + AtSmem::kE + (l + Lk - 1 - r) * kAtPad + d4;
          m0 += er[0]; m1 += er[1]; m2 += er[2]; m3 += er[3];
        }
        a0 = fmaf(w, m0, a0); a1 = fmaf(w, m1, a1); a2 = fmaf(w, m2, a2); a3 = fmaf(w, m3, a3);
      }
      if (live) {
        T* dst = BWD ? dq + (static_cast<size_t>(b) * Lq + q0 + l) * lddq + h * kAtD + d4
                     : out + (static_cast<size_t>(b) * Lq + q0 + l) * H + h * kAtD + d4;
        dst[0] = from_f32<T>(a0); dst[1] = from_f32<T>(a1); dst[2] = from_f32<T>(a2); dst[3] = from_f32<T>(a3);
      }
    }
    if (BWD) {
      // dk_r += sum_l dS[l][r] q_l ; dv_r += sum_l drop(P)[l][r] dO_l : thread (r = t >> 1, feature half = t & 1)
      const int r = t >> 1, hf = (t & 1) * 32;
      for (int ll = 0; ll < kAtQB; ++ll) {
        const float ds = sm[AtSmem::kdS + ll * (kAtMaxK + 1) + r];
        const float pd = sm[AtSmem::kS + ll * (kAtMaxK + 1) + r];
        const float* sq = sm + AtSmem::kQ + ll * kAtPad + hf;
        const float* so = sm + AtSmem::kdO + ll * kAtPad + hf;
#pragma unroll
        for (int d = 0; d < 32; ++d) {
          dkr[d] = fmaf(ds, sq[d], dkr[d]);
          dvr[d] = fmaf(pd, so[d], dvr[d]);
        }
      }
      if (REL) {
        // dE along the diagonals: window row w collects sum_l dS[l][l + Lk - 1 - w] q_l ; CTA buffer row a = q0 + w
        const int d4 = c * 4;
        for (int w = l; w < kAtQB + Lk - 1; w += 16) {
          float e0 = 0.f, e1 = 0.f, e2 = 0.f, e3 = 0.f;
#pragma unroll
          for (int ll = 0; ll < kAtQB; ++ll) {
            const int r2 = ll + Lk - 1 - w;
            if (r2 >= 0 && r2 < Lk) {
              const float ds = sm[AtSmem::kdS + ll * (kAtMaxK + 1) + r2];
              const float* sq = sm + AtSmem::kQ + ll * kAtPad + d4;
              e0 = fmaf(ds, sq[0], e0); e1 = fmaf(ds, sq[1], e1); e2 = fmaf(ds, sq[2], e2); e3 = fmaf(ds, sq[3], e3);
            }
          }
          float* acc = sm + AtSmem::kdE + (q0 + w) * kAtD + d4;  // (w, d4) is owned by exactly one thread
          acc[0] += e0; acc[1] += e1; acc[2] += e2; acc[3] += e3;
        }
      }
    }
  }
  if (BWD) {
    const int r = t >> 1, hf = (t & 1) * 32;
    if (r < Lk) {
      T* dkp = dk + (static_cast<size_t>(b) * Lk + r) * lddk + h * kAtD + hf;
      T* dvp = dv + (static_cast<size_t>(b) * Lk + r) * lddv + h * kAtD + hf;
#pragma unroll
      for (int d = 0; d < 32; ++d) {
        dkp[d] = from_f32<T>(dkr[d]);
        dvp[d] = from_f32<T>(dvr[d]);
      }
    }
    if (REL) {
      __syncthreads();
      const int na = Lq + Lk - 1;  // diagonal a <-> E row a - (Lk - 1) + P - 1
      for (int e = t; e < na * kAtD; e += kAtThreads) {
        const float x = sm[AtSmem::kdE + e];
        if (x != 0.f) atomicAdd(dE + static_cast<size_t>((e >> 6) - (Lk - 1) + P - 1) * kAtD + (e & 63), x);
      }
    }
  }
}

template <typename T, bool REL, bool BWD>
static int launch_at(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* E, int P,
                     const float* mask, DropSpec dr, T* out, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE,
                     cudaStream_t s) {
  auto kfn = attention_train_kernel<T, REL, BWD>;
  const size_t smem = static_cast<size_t>(REL ? (BWD ? AtSmem::kEnd : AtSmem::kdE) : AtSmem::kE) * sizeof(float);
  static bool configured = false;
  if (!configured) {
    SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(AtSmem::kEnd * sizeof(float))));
    configured = true;
  }
  SD_CUDA(launch_k(kfn, dim3(heads, B), dim3(kAtThreads), smem, s, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, E, P, mask, dr, out, dout, dq, lddq, dk,
                   lddk, dv, lddv, dE));
  SD_LAUNCHED(BWD ? "attention_bwd" : "attention_train_fwd", s);
  return SEQDIFF_OK;
}

static int check_at(int B, int heads, int Lq, int Lk, int ldq, int ldk, int ldv, const void* E, int P) {
  SD_CHECK(B > 0 && heads > 0 && Lq > 0 && Lk > 0, "empty attention");
  SD_CHECK(Lk <= kAtMaxK, "training attention: key length is limited to 128 (reference training uses max_seq_len 64 / 128)");
  SD_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0, "row strides must be multiples of 8 elements");
  SD_CHECK(!E || (Lq <= P && Lk <= P && Lq <= kAtMaxK), "relative_key: sequence longer than max_position_embeddings / 128");
  static_assert(AtSmem::kEnd * sizeof(float) <= 232448, "over the 227 KB shared-memory limit");
  return SEQDIFF_OK;
}

template <typename T>
int attention_train_fwd(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                        const float* key_mask, DropSpec dr, T* out, cudaStream_t s) {
  SD_TRY(check_at(B, heads, Lq, Lk, ldq, ldk, ldv, dist_emb, P));
  if (dist_emb)
    return launch_at<T, true, false>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, out, nullptr, nullptr, 0, nullptr, 0, nullptr, 0,
                                     nullptr, s);
  return launch_at<T, false, false>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, out, nullptr, nullptr, 0, nullptr, 0, nullptr, 0,
                                    nullptr, s);
}
template <typename T>
int attention_bwd(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                  const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s) {
  SD_TRY(check_at(B, heads, Lq, Lk, ldq, ldk, ldv, dist_emb, P));
  SD_CHECK(dout && dq && dk && dv && (!dist_emb || dE), "attention_bwd: null argument");
  if (dist_emb)
    return launch_at<T, true, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, nullptr, dout, dq, lddq, dk, lddk, dv, lddv, dE, s);
  return launch_at<T, false, true>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, dr, nullptr, dout, dq, lddq, dk, lddk, dv, lddv, dE, s);
}
#define SD_INST_AT(T)                                                                                                                              \
  template int attention_train_fwd<T>(int, int, int, int, const T*, int, const T*, int, const T*, int, const T*, int, const float*, DropSpec, T*, \
                                      cudaStream_t);                                                                                              \
  template int attention_bwd<T>(int, int, int, int, const T*, int, const T*, int, const T*, int, const T*, int, const float*, DropSpec, const T*, \
                                T*, int, T*, int, T*, int, float*, cudaStream_t)
SD_INST_AT(float);
SD_INST_AT(bf16);
SD_INST_AT(f16);

}  // namespace seqdiff
