// reverse_step.cu -- the discrete reverse-diffusion step, sequence_model/sample.py:120-179
// (sample_p_zs_given_zt_discrete + compute_batched_over0_posterior_distribution), and the training
// q-sample PeptideDiff.apply_aa_noise (model.py:291-311).
//
// Reference arithmetic per residue n of graph b (all fp32, C = 20 classes):
//   p        = softmax(logits[n])                                              sample.py:162
//   post[i,j]= (Qt[b][j,:].x_t[n]) * Qsb[b][i,j] / (Qtb[b][i,:].x_t[n])          sample.py:129-138 (0 -> 1e-6)
//   un[j]    = sum_i p[i] * post[i,j]      (product rounded, then summed over i) sample.py:165-166
//   un[:]    = 1e-5 if sum_j un[j] == 0;  prob = un / sum_j un                   sample.py:167-168
//   x_s      = multinomial(prob) = argmax_j prob[j] / E[j], E ~ Exp(1)  |  argmax_j prob[j]   sample.py:169-177
// The reference materialises three [N,20,20] tensors and loops over N rows in Python.  Here one CTA
// owns one graph: the (Qt,Qsb,Qtb) triple is staged in shared memory, the 20x20x20 table
// post_x[i,j] for every possible one-hot x_t is built once per CTA with the SAME rounding sequence
// (mul, then IEEE divide), and each thread then resolves one residue with 400 multiply-adds.
// Rows of x_t that are not exactly one-hot take the general (dot-product) formula.
// Traffic: 80 B logits + 80 B x_t in, 80 B one-hot out per residue (+80 B if the noise E is supplied).
//
// Two arithmetic modes (template FAST), same algorithm:
//   exact (noise_E supplied = a reference noise stream is being replayed, or argmax): the reference's own op sequence --
//         expf, IEEE divides, product rounded then summed over i -- so indices agree bit for bit up to libm ulps;
//   fast  (in-kernel Philox noise = production): there is no reference stream to reproduce, only a distribution, so the
//         posterior uses FMA, ex2/lg2/rcp.approx and 128-bit table loads, and skips the two normalisations (an argmax race is
//         invariant to positive row scaling).  Deviation of the race scores <= ~3e-6 relative (pinned: tests/test_gpu_ops.py::test_reverse_step_philox_pinned_to_oracle).  ncu (round 1): the exact path
//         costs 5075 thread-instructions per residue at 63 % issue utilisation -- the kernel is issue-bound, not HBM-bound.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

namespace seqdiff {

constexpr int C = SEQDIFF_NUM_CLASSES;
constexpr int kRevThreads = 256;

// raw words for (graph, residue-in-graph, step): class j uses word j%4 of call j/4.
// counter = (residue, step*8 + call, graph_lo, graph_hi), key = seed.
__device__ __forceinline__ void philox_row(uint64_t seed, uint64_t graph, uint32_t residue, uint32_t step, uint32_t (&w)[C]) {
#pragma unroll
  for (int call = 0; call < C / 4; ++call) {
    uint32_t c[4] = {residue, step * 8u + call, static_cast<uint32_t>(graph), static_cast<uint32_t>(graph >> 32)};
    philox4x32_10(c, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
#pragma unroll
    for (int i = 0; i < 4; ++i) w[call * 4 + i] = c[i];
  }
}
// u in (0,1) exactly representable: ((w >> 9) + 0.5) * 2^-23 ;  E = -log(u) > 0
__device__ __forceinline__ float exp1_from_u32(uint32_t w) {
  const float u = (static_cast<float>(w >> 9) + 0.5f) * 1.1920928955078125e-07f;
  return -logf(u);
}
__device__ __forceinline__ float lg2_approx(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// 1 / (-log2 u): the Exp(1) variate up to the constant ln 2, inverted (the race only compares ratios).
// lg2.approx has an ABSOLUTE error of 2^-22 on (0.5, 2), so near u = 1 (where -log2 u -> 0) its relative error explodes and the
// result can even be 0 or change sign.  For v = 1 - u < 1/8 (exactly representable: u has 24 significant bits) the series
//   -log2(1 - v) = log2(e) * v * (1 + v/2 + v^2/3 + ... + v^6/7)          (truncation < v^7/8 < 6e-8 relative)
// is used instead; for v >= 1/8 the magnitude of lg2 is >= 0.19, i.e. <= 1.3e-6 relative.  Branch-free (select).
__device__ __forceinline__ float inv_exp1_fast(uint32_t w) {
  const float u = (static_cast<float>(w >> 9) + 0.5f) * 1.1920928955078125e-07f;
  const float v = 1.0f - u;
  float ser = fmaf(v, 1.0f / 7.0f, 1.0f / 6.0f);
  ser = fmaf(ser, v, 0.2f);
  ser = fmaf(ser, v, 0.25f);
  ser = fmaf(ser, v, 1.0f / 3.0f);
  ser = fmaf(ser, v, 0.5f);
  ser = fmaf(ser, v, 1.0f);
  const float near1 = ser * v * 1.44269504088896f;
  const float e2 = v < 0.125f ? near1 : -lg2_approx(u);
  return rcp_approx(e2);
}

// two fp32 FMAs in one instruction (FFMA2 on sm_100a): d = a * b + c on both halves.  Same rounding as two fmaf.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t ra, rb, rc, rd;
  ra = *reinterpret_cast<uint64_t*>(&a); rb = *reinterpret_cast<uint64_t*>(&b); rc = *reinterpret_cast<uint64_t*>(&c);
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return *reinterpret_cast<float2*>(&rd);
}

// exponential race / argmax over one normalised row
__device__ __forceinline__ int pick_class(const float (&prob)[C], bool diverse, const float (&E)[C]) {
  int best = 0;
  float bv = -INFINITY;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    const float v = diverse ? __fdiv_rn(prob[j], E[j]) : prob[j];
    if (v > bv) { bv = v; best = j; }  // first maximum wins, like torch.argmax
  }
  return best;
}

__device__ __forceinline__ void write_onehot(float* __restrict__ row, int idx) {
#pragma unroll
  for (int j4 = 0; j4 < C; j4 += 4) {
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (idx == j4) o.x = 1.f;
    if (idx == j4 + 1) o.y = 1.f;
    if (idx == j4 + 2) o.z = 1.f;
    if (idx == j4 + 3) o.w = 1.f;
    *reinterpret_cast<float4*>(row + j4) = o;
  }
}

// The same shared-memory pointer, with its address computed at run time (shared window -> generic).  The fast kernel passes its tables
// through this to the cold-path helper below: with one caller left, the compiler would otherwise specialise the helper on the three
// static table addresses, and that shifts the caller's register allocation into 88 B of spills.
__device__ __forceinline__ const float* opaque_smem(const float* p) {
  return static_cast<const float*>(__cvta_shared_to_generic(__cvta_generic_to_shared(p)));
}

// Cold path: a row of x_t that is not exactly one-hot (never produced by the sampler itself; sample.py:129-138 accepts it).
// Kept out of line and fed from global/shared memory so that the hot path's per-class arrays stay in registers.
//   left[j] = Qt[j,:].x ; den[i] = Qtb[i,:].x (0 -> 1e-6) ; un[j] = sum_i p_i * left[j] * Qsb[i,j] / den[i]
template <bool FAST>
__device__ __noinline__ int soft_row_class(const float* __restrict__ lg_row, const float* x_row, const float* sQt,
                                           const float* sQsb, const float* sQtb, bool diverse, const float* __restrict__ E_row, uint64_t seed,
                                           uint64_t graph, uint32_t l, uint32_t step) {
  float mx = lg_row[0];
  for (int j = 1; j < C; ++j) mx = fmaxf(mx, lg_row[j]);
  float ps = 0.f;
  for (int j = 0; j < C; ++j) ps += expf(lg_row[j] - mx);
  float un[C];
#pragma unroll
  for (int j = 0; j < C; ++j) un[j] = 0.f;
  for (int i = 0; i < C; ++i) {
    const float p = __fdiv_rn(expf(lg_row[i] - mx), ps);
    float den = 0.f;
    for (int k = 0; k < C; ++k) den = fmaf(sQtb[i * C + k], x_row[k], den);
    if (den == 0.f) den = 1e-6f;
#pragma unroll
    for (int j = 0; j < C; ++j) {
      float left = 0.f;
      for (int k = 0; k < C; ++k) left = fmaf(x_row[k], sQt[j * C + k], left);
      un[j] = __fadd_rn(un[j], __fmul_rn(p, __fdiv_rn(__fmul_rn(left, sQsb[i * C + j]), den)));
    }
  }
  float tot = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) tot += un[j];
  if (tot == 0.f) {
    tot = 0.f;
#pragma unroll
    for (int j = 0; j < C; ++j) { un[j] = 1e-5f; tot += 1e-5f; }
  }
  uint32_t w[C];
  if (diverse && !E_row) philox_row(seed, graph, l, step, w);
  int best = 0;
  float bv = -INFINITY, psum = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    const float pr = __fdiv_rn(un[j], tot);
    psum += pr;
    const float v = !diverse ? pr : (E_row ? __fdiv_rn(pr, E_row[j]) : (FAST ? pr * inv_exp1_fast(w[j]) : __fdiv_rn(pr, exp1_from_u32(w[j]))));
    if (v > bv) { bv = v; best = j; }
  }
  return psum != 0.f ? best : 0;
}

template <bool FAST, int THREADS = kRevThreads, int MINB = (FAST ? 2 : 1)>
__global__ void __launch_bounds__(THREADS, MINB) reverse_step_kernel(const float* __restrict__ q_tables, int n_tab, int L,
                                                                   const float* x_t, const float* __restrict__ logits,
                                                                   int diverse, const float* __restrict__ noise_E, uint64_t seed,
                                                                   uint64_t graph_id0, uint32_t step, const int* __restrict__ step_ptr,
                                                                   float* x_s, uint8_t* __restrict__ idx_out, int* __restrict__ advance,
                                                                   const uint64_t* __restrict__ rng) {
  // x_t / x_s carry no __restrict__: the sampling loop runs the step IN PLACE (x_s == x_t; each thread reads its own row
  // completely before it writes it -- the contract documented in kernels.h).
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  if (rng) {  // sampling loop: (seed, first global graph id) live in device memory so that a cached CUDA graph serves every call
    seed = rng[0];
    graph_id0 = rng[1];
  }
  __shared__ float sQt[C * C], sQsb[C * C], sQtb[C * C];
  // exact mode: post[x][i][j] = Qt[j,x] Qsb[i,j] / Qtb[i,x] with the reference's rounding sequence, odd x-stride (401: lanes
  // holding different x_t classes read 32 different banks; stride 400 folded all classes onto 2 banks -- 16-way conflicts).
  // fast mode never builds that 32 KB table (its 8000-entry build per CTA and its 1.6 KB of lane-private smem reads per
  // residue were the bound: 20 us per 131072 residues).  It factors the posterior as
  //     un[j] = Qt[j,x] * sum_i (p_i / Qtb[i,x]) * Qsb[i,j]
  // so the 400-term inner product reads Qsb only -- the SAME address in every lane (smem broadcast) -- and the two
  // x-dependent factors are one 20-float row each of the transposed tables InvT[x][i] = 1 / Qtb[i,x], QtT[x][j] = Qt[j,x].
  constexpr int kXS = C * C + 1;
  constexpr int kRS = C + 4;  // row stride of the transposed tables: rows stay 16 B aligned
  __shared__ float sPost[FAST ? 1 : C * kXS];
  __shared__ __align__(16) float sInvT[FAST ? C * kRS : 4], sQtT[FAST ? C * kRS : 4];
  __shared__ __align__(16) float sQsbA[FAST ? C * C : 4];  // 16 B aligned copy of Qsb for 128-bit broadcast reads
  const int b = blockIdx.y;  // grid = (ceil(L / 128) residue chunks, graphs): enough CTAs to stream at HBM rate
  const size_t n_res = static_cast<size_t>(gridDim.y) * L;
  if (step_ptr) {
    // one read of the step counter per CTA (thread 0), shared through smem; with `advance` the CTA that is last to have
    // read it moves the counter on to the next step -- no CTA can still be about to read the old value then
    __shared__ int s_sidx;
    if (threadIdx.x == 0) {
      s_sidx = *reinterpret_cast<const volatile int*>(step_ptr);
      if (advance) {
        __threadfence();
        const unsigned total = gridDim.x * gridDim.y;
        if (atomicAdd(reinterpret_cast<unsigned*>(advance), 1u) == total - 1u) {
          *reinterpret_cast<volatile unsigned*>(advance) = 0u;
          *const_cast<int*>(step_ptr) = s_sidx - 1;
        }
      }
    }
    __syncthreads();
    const int sidx = s_sidx;
    SD_DEV_ASSERT(sidx >= 0);  // the loop counter never runs past the last step
    if (sidx == 0) return;  // last step: caller keeps the raw logits (sample.py:147-148)
    step = static_cast<uint32_t>(sidx);
    q_tables += static_cast<size_t>(sidx) * (3 * C * C);
    if (noise_E) noise_E += static_cast<size_t>(sidx) * n_res * C;
  }
  const float* tab = q_tables + static_cast<size_t>(n_tab == 1 ? 0 : b) * (3 * C * C);
  for (int i = threadIdx.x; i < C * C; i += THREADS) {
    sQt[i] = tab[i];
    sQsb[i] = tab[C * C + i];
    sQtb[i] = tab[2 * C * C + i];
  }
  __syncthreads();
  if (FAST) {
    for (int e = threadIdx.x; e < C * C; e += THREADS) {
      const int r = e / C, x = e - r * C;  // r = i for Qtb[i,x], r = j for Qt[j,x]
      const float den = sQtb[e];
      sInvT[x * kRS + r] = rcp_approx(den == 0.f ? 1e-6f : den);
      sQtT[x * kRS + r] = sQt[e];
      sQsbA[e] = sQsb[e];
    }
  } else {
    for (int e = threadIdx.x; e < C * C; e += THREADS) {  // (i, j) fixed per thread, x runs: no div/mod in the inner loop
      const int i = e / C, j = e - i * C;
      const float qsb = sQsb[e];
#pragma unroll 4
      for (int x = 0; x < C; ++x) {
        float den = sQtb[i * C + x];
        if (den == 0.f) den = 1e-6f;
        sPost[x * kXS + e] = __fdiv_rn(__fmul_rn(sQt[j * C + x], qsb), den);
      }
    }
  }
  __syncthreads();

  if (FAST) {
    // Production path.  A thread resolves RJ = 2 residues JOINTLY (l and l + THREADS of its CTA's slab): every 128-bit broadcast read
    // of Qsb feeds the FFMA2s of both, and the two softmax / Philox / race chains are independent instruction streams for the
    // scheduler -- the kernel is bound by dependency latency (41 % issue utilisation with one chain per thread, DESIGN.md section 9),
    // not by HBM or a pipe.  A residue past L is computed on clamped inputs and not stored.
    constexpr int RJ = 2;
    const float4* qsb4 = reinterpret_cast<const float4*>(sQsbA);
    const uint64_t graph = graph_id0 + b;
    for (int l0 = blockIdx.x * (RJ * THREADS) + threadIdx.x; l0 < L; l0 += gridDim.x * (RJ * THREADS)) {
      asm volatile("" ::: "memory");  // keeps the 100 broadcast reads of Qsb inside the iteration (hoisted out of the loop they spill: 1.6 KB of stack)
      int lr[RJ];
      bool live[RJ];
      size_t nr[RJ];
#pragma unroll
      for (int r = 0; r < RJ; ++r) {
        const int l = l0 + r * THREADS;
        live[r] = l < L;
        lr[r] = live[r] ? l : l0;
        nr[r] = static_cast<size_t>(b) * L + lr[r];
      }
      float pf[RJ][C];
      int hotf[RJ];
      bool onehot[RJ];
#pragma unroll
      for (int r = 0; r < RJ; ++r) {
        float xr[C];
#pragma unroll
        for (int j4 = 0; j4 < C; j4 += 4) {
          const float4 a = *reinterpret_cast<const float4*>(logits + nr[r] * C + j4);
          const float4 c4 = *reinterpret_cast<const float4*>(x_t + nr[r] * C + j4);
          pf[r][j4] = a.x; pf[r][j4 + 1] = a.y; pf[r][j4 + 2] = a.z; pf[r][j4 + 3] = a.w;
          xr[j4] = c4.x; xr[j4 + 1] = c4.y; xr[j4 + 2] = c4.z; xr[j4 + 3] = c4.w;
        }
        int h = -1, nnz = 0;
#pragma unroll
        for (int j = 0; j < C; ++j)
          if (xr[j] != 0.f) { ++nnz; h = (xr[j] == 1.0f) ? j : -2; }
        onehot[r] = nnz == 1 && h >= 0;
        hotf[r] = onehot[r] ? h : 0;
      }
#pragma unroll
      for (int r = 0; r < RJ; ++r) {
        float mxf = pf[r][0];
#pragma unroll
        for (int j = 1; j < C; ++j) mxf = fmaxf(mxf, pf[r][j]);
#pragma unroll
        for (int j = 0; j < C; ++j) pf[r][j] = ex2_approx((pf[r][j] - mxf) * 1.44269504088896f);  // unnormalised softmax
        const float4* inv4 = reinterpret_cast<const float4*>(sInvT + hotf[r] * kRS);
#pragma unroll
        for (int i4 = 0; i4 < C / 4; ++i4) {  // a_i = p_i / Qtb[i,x]
          const float4 w = inv4[i4];
          pf[r][4 * i4] *= w.x; pf[r][4 * i4 + 1] *= w.y; pf[r][4 * i4 + 2] *= w.z; pf[r][4 * i4 + 3] *= w.w;
        }
      }
      float2 un2[RJ][C / 2];
#pragma unroll
      for (int r = 0; r < RJ; ++r)
#pragma unroll
        for (int j = 0; j < C / 2; ++j) un2[r][j] = make_float2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < C; ++i) {  // fully unrolled: pf[.][i] must stay in registers
#pragma unroll
        for (int j4 = 0; j4 < C / 4; ++j4) {
          const float4 w = qsb4[i * (C / 4) + j4];  // same address in every lane: broadcast; one read serves both residues
#pragma unroll
          for (int r = 0; r < RJ; ++r) {
            const float2 pp = make_float2(pf[r][i], pf[r][i]);
            un2[r][2 * j4] = ffma2(pp, make_float2(w.x, w.y), un2[r][2 * j4]);          // FFMA2: 200 instead of 400 FMA issues per residue
            un2[r][2 * j4 + 1] = ffma2(pp, make_float2(w.z, w.w), un2[r][2 * j4 + 1]);
          }
        }
      }
      int best[RJ];
      float bv[RJ];
#pragma unroll
      for (int r = 0; r < RJ; ++r) {
        const float4* qt4 = reinterpret_cast<const float4*>(sQtT + hotf[r] * kRS);
        float totf = 0.f;
#pragma unroll
        for (int j4 = 0; j4 < C / 4; ++j4) {
          const float4 w = qt4[j4];
          un2[r][2 * j4].x *= w.x; un2[r][2 * j4].y *= w.y; un2[r][2 * j4 + 1].x *= w.z; un2[r][2 * j4 + 1].y *= w.w;
          totf += (un2[r][2 * j4].x + un2[r][2 * j4].y) + (un2[r][2 * j4 + 1].x + un2[r][2 * j4 + 1].y);
        }
        if (totf == 0.f) {  // sample.py:167: all-zero row -> uniform
#pragma unroll
          for (int j = 0; j < C / 2; ++j) un2[r][j] = make_float2(1e-5f, 1e-5f);
        }
        best[r] = 0;
        bv[r] = -INFINITY;
      }
      // race: class j uses word j % 4 of Philox call j / 4 (same stream as philox_row); one call per residue at a time so that only
      // 2 x 4 words are live, winners of each group of 4 found by a 2-level tree, groups folded in order (first maximum wins, as argmax)
#pragma unroll
      for (int call = 0; call < C / 4; ++call) {
#pragma unroll
        for (int r = 0; r < RJ; ++r) {
          uint32_t c4[4] = {static_cast<uint32_t>(lr[r]), step * 8u + call, static_cast<uint32_t>(graph), static_cast<uint32_t>(graph >> 32)};
          philox4x32_10(c4, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
          const float v0 = un2[r][2 * call].x * inv_exp1_fast(c4[0]), v1 = un2[r][2 * call].y * inv_exp1_fast(c4[1]);
          const float v2 = un2[r][2 * call + 1].x * inv_exp1_fast(c4[2]), v3 = un2[r][2 * call + 1].y * inv_exp1_fast(c4[3]);
          const bool a = v1 > v0, c = v3 > v2;
          const float va = a ? v1 : v0, vc = c ? v3 : v2;
          const int ia = 4 * call + (a ? 1 : 0), ic = 4 * call + (c ? 3 : 2);
          const bool e = vc > va;
          const float vg = e ? vc : va;
          const int ig = e ? ic : ia;
          if (vg > bv[r]) { bv[r] = vg; best[r] = ig; }
        }
      }
#pragma unroll
      for (int r = 0; r < RJ; ++r) {
        if (!live[r]) continue;
        int idx = best[r];
        if (!onehot[r])  // cold: a row of x_t that is not exactly one-hot (never produced by the sampler itself)
          idx = soft_row_class<true>(logits + nr[r] * C, x_t + nr[r] * C, opaque_smem(sQt), opaque_smem(sQsb), opaque_smem(sQtb), true, nullptr, seed, graph,
                                     static_cast<uint32_t>(lr[r]), step);
        write_onehot(x_s + nr[r] * C, idx);
        if (idx_out) idx_out[nr[r]] = static_cast<uint8_t>(idx);
      }
    }
    return;
  }
  for (int l = blockIdx.x * THREADS + threadIdx.x; l < L; l += gridDim.x * THREADS) {
    const size_t n = static_cast<size_t>(b) * L + l;
    float lg[C], xr[C];
#pragma unroll
    for (int j4 = 0; j4 < C; j4 += 4) {
      const float4 a = *reinterpret_cast<const float4*>(logits + n * C + j4);
      const float4 c4 = *reinterpret_cast<const float4*>(x_t + n * C + j4);
      lg[j4] = a.x; lg[j4 + 1] = a.y; lg[j4 + 2] = a.z; lg[j4 + 3] = a.w;
      xr[j4] = c4.x; xr[j4 + 1] = c4.y; xr[j4 + 2] = c4.z; xr[j4 + 3] = c4.w;
    }
    if (FAST) continue;  // (the production path is the joint loop above)
    // softmax(logits)
    float mx = lg[0];
#pragma unroll
    for (int j = 1; j < C; ++j) mx = fmaxf(mx, lg[j]);
    float p[C], ps = 0.f;
#pragma unroll
    for (int j = 0; j < C; ++j) { p[j] = expf(lg[j] - mx); ps += p[j]; }
#pragma unroll
    for (int j = 0; j < C; ++j) p[j] = __fdiv_rn(p[j], ps);
    // one-hot?
    int hot = -1, nnz = 0;
#pragma unroll
    for (int j = 0; j < C; ++j)
      if (xr[j] != 0.f) { ++nnz; hot = (xr[j] == 1.0f) ? j : -2; }
    float un[C];
#pragma unroll
    for (int j = 0; j < C; ++j) un[j] = 0.f;
    if (nnz == 1 && hot >= 0) {
      const float* post = sPost + hot * kXS;
#pragma unroll
      for (int i = 0; i < C; ++i) {
#pragma unroll
        for (int j = 0; j < C; ++j) un[j] = __fadd_rn(un[j], __fmul_rn(p[i], post[i * C + j]));
      }
    } else {
      const int idx = soft_row_class<false>(logits + n * C, x_t + n * C, sQt, sQsb, sQtb, diverse != 0, noise_E ? noise_E + n * C : nullptr, seed,
                                            graph_id0 + b, static_cast<uint32_t>(l), step);
      write_onehot(x_s + n * C, idx);
      if (idx_out) idx_out[n] = static_cast<uint8_t>(idx);
      continue;
    }
    float tot = 0.f;
#pragma unroll
    for (int j = 0; j < C; ++j) tot += un[j];
    if (tot == 0.f) {
      tot = 0.f;
#pragma unroll
      for (int j = 0; j < C; ++j) { un[j] = 1e-5f; tot += 1e-5f; }
    }
    float prob[C], psum = 0.f;
#pragma unroll
    for (int j = 0; j < C; ++j) { prob[j] = __fdiv_rn(un[j], tot); psum += prob[j]; }
    float E[C];
    if (diverse) {
      if (noise_E) {
#pragma unroll
        for (int j4 = 0; j4 < C; j4 += 4) {
          const float4 a = *reinterpret_cast<const float4*>(noise_E + n * C + j4);
          E[j4] = a.x; E[j4 + 1] = a.y; E[j4 + 2] = a.z; E[j4 + 3] = a.w;
        }
      } else {
        uint32_t w[C];
        philox_row(seed, graph_id0 + b, static_cast<uint32_t>(l), step, w);
#pragma unroll
        for (int j = 0; j < C; ++j) E[j] = exp1_from_u32(w[j]);
      }
    }
    int idx = 0;
    if (psum != 0.f) idx = pick_class(prob, diverse != 0, E);
    write_onehot(x_s + n * C, idx);
    if (idx_out) idx_out[n] = static_cast<uint8_t>(idx);
  }
}

int reverse_step(const float* q_tables, int n_tab, int B, int L, const float* x_t, const float* logits, int diverse,
                 const float* noise_E, uint64_t seed, uint64_t graph_id0, uint32_t step, const int* step_ptr, float* x_s,
                 uint8_t* idx_out, cudaStream_t s, int* advance, const uint64_t* rng) {
  SD_CHECK(B > 0 && L > 0, "empty reverse step");
  SD_CHECK(n_tab == 1 || n_tab == B, "q_tables must hold 1 or B (Qt,Qsb,Qtb) triples");
  // 256 threads per CTA, 2 residues per thread; the fast kernel with 2 CTAs per SM (launch-shape sweep on B200: profiles/revstep_r01.log)
  const dim3 grid(ceil_div(L, 2 * kRevThreads), B);
  if (diverse && !noise_E)
    SD_CUDA(launch_k(reverse_step_kernel<true, 256, 2>, dim3(grid), dim3(kRevThreads), 0, s, q_tables, n_tab, L, x_t, logits, diverse, noise_E, seed, graph_id0, step, step_ptr, x_s, idx_out, advance, rng));
  else
    SD_CUDA(launch_k(reverse_step_kernel<false>, dim3(grid), dim3(kRevThreads), 0, s, q_tables, n_tab, L, x_t, logits, diverse, noise_E, seed, graph_id0, step, step_ptr, x_s, idx_out, advance, rng));
  SD_LAUNCHED("reverse_step", s);
  return SEQDIFF_OK;
}

// ---------------------------------------------------------------------------------------------------
// q-sample (training): prob[i] = Qtb[b][i,:].x0[n]; all-zero rows (padding) -> class 0  (model.py:301-308)
// step_ptr != NULL (the scoring loop): every graph draws from the step's Qtb = q_tables[k][2] (qtb = the [T,3,20,20] step tables),
// k = *step_ptr (read only: the step's last kernel advances it), noise entry k of a [T, B*L, 20] noise_E, (seed, graph_id0) from rng.
__global__ void __launch_bounds__(kRevThreads) apply_aa_noise_kernel(const float* __restrict__ qtb, int L, const float* __restrict__ x0,
                                                                     const float* __restrict__ noise_E, uint64_t seed, uint64_t graph_id0,
                                                                     uint32_t step, float* __restrict__ x_t, uint8_t* __restrict__ idx_out,
                                                                     const int* __restrict__ step_ptr, const uint64_t* __restrict__ rng) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  __shared__ float sQ[C * C];
  const int b = blockIdx.x;
  size_t tab = static_cast<size_t>(b) * C * C;
  if (step_ptr) {
    const int k = *step_ptr;
    SD_DEV_ASSERT(k >= 0);
    tab = static_cast<size_t>(k) * (3 * C * C) + 2 * C * C;
    step = static_cast<uint32_t>(k);
    if (noise_E) noise_E += static_cast<size_t>(k) * gridDim.x * L * C;
    seed = rng[0];
    graph_id0 = rng[1];
  }
  for (int i = threadIdx.x; i < C * C; i += kRevThreads) sQ[i] = qtb[tab + i];
  __syncthreads();
  for (int l = threadIdx.x; l < L; l += kRevThreads) {
    const size_t n = static_cast<size_t>(b) * L + l;
    float xr[C];
#pragma unroll
    for (int j4 = 0; j4 < C; j4 += 4) {
      const float4 c4 = *reinterpret_cast<const float4*>(x0 + n * C + j4);
      xr[j4] = c4.x; xr[j4 + 1] = c4.y; xr[j4 + 2] = c4.z; xr[j4 + 3] = c4.w;
    }
    // one-hot row (what the dataset holds): prob[i] = Qtb[i, hot] -- a column read, the same value the dot product gives
    // (1 * q + 0 * ... exactly); anything else takes the general dot product.  (The fully unrolled 400-term form for every row
    // needed 255 registers and 792 B of spills.)
    int hot = -1, nnz = 0;
#pragma unroll
    for (int k = 0; k < C; ++k)
      if (xr[k] != 0.f) { ++nnz; hot = (xr[k] == 1.0f) ? k : -2; }
    float prob[C], psum = 0.f;
    if (nnz == 1 && hot >= 0) {
#pragma unroll
      for (int i = 0; i < C; ++i) {
        prob[i] = sQ[i * C + hot];
        psum += prob[i];
      }
    } else {
#pragma unroll 1
      for (int i = 0; i < C; ++i) {
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < C; ++k) a = fmaf(sQ[i * C + k], xr[k], a);
        prob[i] = a;
        psum += a;
      }
    }
    int idx = 0;
    if (psum != 0.f) {
      float E[C];
      if (noise_E) {
#pragma unroll
        for (int j = 0; j < C; ++j) E[j] = noise_E[n * C + j];
      } else {
        uint32_t w[C];
        philox_row(seed, graph_id0 + b, static_cast<uint32_t>(l), step, w);
#pragma unroll
        for (int j = 0; j < C; ++j) E[j] = exp1_from_u32(w[j]);
      }
      idx = pick_class(prob, true, E);
    }
    write_onehot(x_t + n * C, idx);
    if (idx_out) idx_out[n] = static_cast<uint8_t>(idx);
  }
}

int apply_aa_noise(const float* qtb, int B, int L, const float* x0, const float* noise_E, uint64_t seed, uint64_t graph_id0,
                   uint32_t step, float* x_t, uint8_t* idx_out, cudaStream_t s, const int* step_ptr, const uint64_t* rng) {
  SD_CHECK(B > 0 && L > 0, "empty q-sample");
  SD_CHECK(!step_ptr || rng, "the in-loop q-sample reads its Philox key from device memory");
  SD_CUDA(launch_k(apply_aa_noise_kernel, dim3(B), dim3(kRevThreads), 0, s, qtb, L, x0, noise_E, seed, graph_id0, step, x_t, idx_out, step_ptr, rng));
  SD_LAUNCHED("apply_aa_noise", s);
  return SEQDIFF_OK;
}

// ---------------------------------------------------------------------------------------------------
// Terms of the variational bound at step k of the scoring loop (Model::score), one thread per residue n of graph b, valid ones only:
//   ce  = -log softmax(z)_a                                    (a = native class: x0 one-hot, z = the step's logits; fp64 from fp32 z)
//   k >= 1: kl = sum_{j: q_j > 0} q_j (log q_j - log max(p_j, 1e-30))  in fp64, where
//           p = the reverse step's normalised prob (exact mode above: softmax, sPost with the reference's rounding, 1e-5 rows) and
//           q = the same with one-hot(a) for softmax(z), i.e. row a of post_x normalised   (x = the drawn class of x_t)
//   k == 0: kl is replaced by the reconstruction term ce (the step at which the sampler returns the raw logits)
// acc[n] += (kl or ce, ce).  A thread owns its residue's two fp64 sums and the steps run in sequence: bit-reproducible sums.
// The step counter is read and advanced as in reverse_step_kernel (advance / step_ptr).
constexpr int kVlbThreads = 128;
__global__ void __launch_bounds__(kVlbThreads) vlb_terms_kernel(const float* __restrict__ q_tables, int L, const float* __restrict__ x0,
                                                                const float* __restrict__ x_t, const float* __restrict__ logits,
                                                                const float* __restrict__ mask, const int* __restrict__ step_ptr,
                                                                int* __restrict__ advance, double* __restrict__ acc) {
  pdl_trigger();
  pdl_wait();
  __shared__ int s_sidx;
  if (threadIdx.x == 0) {
    s_sidx = *reinterpret_cast<const volatile int*>(step_ptr);
    __threadfence();
    const unsigned total = gridDim.x * gridDim.y;
    if (atomicAdd(reinterpret_cast<unsigned*>(advance), 1u) == total - 1u) {
      *reinterpret_cast<volatile unsigned*>(advance) = 0u;
      *const_cast<int*>(step_ptr) = s_sidx - 1;
    }
  }
  __syncthreads();
  const int k = s_sidx;
  SD_DEV_ASSERT(k >= 0);
  constexpr int kXS = C * C + 1;  // odd x-stride, as in the exact reverse step
  __shared__ float sQt[C * C], sQsb[C * C], sQtb[C * C];
  __shared__ float sPost[C * kXS];
  if (k > 0) {
    const float* tab = q_tables + static_cast<size_t>(k) * (3 * C * C);
    for (int i = threadIdx.x; i < C * C; i += kVlbThreads) {
      sQt[i] = tab[i];
      sQsb[i] = tab[C * C + i];
      sQtb[i] = tab[2 * C * C + i];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < C * C; e += kVlbThreads) {
      const int i = e / C, j = e - i * C;
      const float qsb = sQsb[e];
      for (int x = 0; x < C; ++x) {
        float den = sQtb[i * C + x];
        if (den == 0.f) den = 1e-6f;
        sPost[x * kXS + e] = __fdiv_rn(__fmul_rn(sQt[j * C + x], qsb), den);
      }
    }
    __syncthreads();
  }
  const int b = blockIdx.y;
  for (int l = blockIdx.x * kVlbThreads + threadIdx.x; l < L; l += gridDim.x * kVlbThreads) {
    const size_t n = static_cast<size_t>(b) * L + l;
    if (mask[n] == 0.f) continue;
    float lg[C];
    int a = -1, x = -1;
#pragma unroll
    for (int j4 = 0; j4 < C; j4 += 4) {
      const float4 z = *reinterpret_cast<const float4*>(logits + n * C + j4);
      const float4 t = *reinterpret_cast<const float4*>(x0 + n * C + j4);
      const float4 d = *reinterpret_cast<const float4*>(x_t + n * C + j4);
      lg[j4] = z.x; lg[j4 + 1] = z.y; lg[j4 + 2] = z.z; lg[j4 + 3] = z.w;
      if (t.x != 0.f) a = j4; if (t.y != 0.f) a = j4 + 1; if (t.z != 0.f) a = j4 + 2; if (t.w != 0.f) a = j4 + 3;
      if (d.x != 0.f) x = j4; if (d.y != 0.f) x = j4 + 1; if (d.z != 0.f) x = j4 + 2; if (d.w != 0.f) x = j4 + 3;
    }
    SD_DEV_ASSERT(a >= 0 && x >= 0);  // valid rows of x0 are one-hot (checked by the caller); x_t is the q-sample's one-hot
    float mx = lg[0];
#pragma unroll
    for (int j = 1; j < C; ++j) mx = fmaxf(mx, lg[j]);
    double se = 0.0;
#pragma unroll
    for (int j = 0; j < C; ++j) se += exp(static_cast<double>(lg[j]) - static_cast<double>(mx));
    const double ce = log(se) - (static_cast<double>(lg[a]) - static_cast<double>(mx));
    double t0 = ce;
    if (k > 0) {
      float p[C], ps = 0.f;
#pragma unroll
      for (int j = 0; j < C; ++j) { p[j] = expf(lg[j] - mx); ps += p[j]; }
#pragma unroll
      for (int j = 0; j < C; ++j) p[j] = __fdiv_rn(p[j], ps);
      const float* post = sPost + x * kXS;
      float un[C];
#pragma unroll
      for (int j = 0; j < C; ++j) un[j] = 0.f;
#pragma unroll
      for (int i = 0; i < C; ++i) {
#pragma unroll
        for (int j = 0; j < C; ++j) un[j] = __fadd_rn(un[j], __fmul_rn(p[i], post[i * C + j]));
      }
      float tot = 0.f, totq = 0.f;
#pragma unroll
      for (int j = 0; j < C; ++j) { tot += un[j]; totq += post[a * C + j]; }
      const bool pz = tot == 0.f, qz = totq == 0.f;
      float tz = 0.f;  // sample.py:167: an all-zero row becomes 1e-5 everywhere, summed in order as in the reverse step
#pragma unroll
      for (int j = 0; j < C; ++j) tz += 1e-5f;
      if (pz) tot = tz;
      if (qz) totq = tz;
      double kl = 0.0;
#pragma unroll
      for (int j = 0; j < C; ++j) {
        const float pj = __fdiv_rn(pz ? 1e-5f : un[j], tot);
        const float qj = __fdiv_rn(qz ? 1e-5f : post[a * C + j], totq);
        if (qj > 0.f) kl += static_cast<double>(qj) * (log(static_cast<double>(qj)) - log(static_cast<double>(fmaxf(pj, 1e-30f))));
      }
      t0 = kl;
    }
    acc[2 * n] += t0;
    acc[2 * n + 1] += ce;
  }
}

int vlb_terms(const float* q_tables, int B, int L, const float* x0, const float* x_t, const float* logits, const float* mask,
              const int* step_ptr, int* advance, double* acc, cudaStream_t s) {
  SD_CHECK(B > 0 && L > 0, "empty score step");
  SD_CHECK(step_ptr && advance, "the score step is indexed by the loop's device step counter");
  SD_CUDA(launch_k(vlb_terms_kernel, dim3(ceil_div(L, kVlbThreads), B), dim3(kVlbThreads), 0, s, q_tables, L, x0, x_t, logits, mask, step_ptr,
                   advance, acc));
  SD_LAUNCHED("vlb_terms", s);
  return SEQDIFF_OK;
}

__global__ void philox_u32_kernel(uint64_t seed, uint64_t graph_id0, uint32_t step, int L, uint32_t* __restrict__ out) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  const int b = blockIdx.x;
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    uint32_t w[C];
    philox_row(seed, graph_id0 + b, static_cast<uint32_t>(l), step, w);
    for (int j = 0; j < C; ++j) out[(static_cast<size_t>(b) * L + l) * C + j] = w[j];
  }
}
int philox_u32(uint64_t seed, uint64_t graph_id0, uint32_t step, int B, int L, uint32_t* out, cudaStream_t s) {
  SD_CUDA(launch_k(philox_u32_kernel, dim3(B), dim3(128), 0, s, seed, graph_id0, step, L, out));
  SD_LAUNCHED("philox_u32", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
