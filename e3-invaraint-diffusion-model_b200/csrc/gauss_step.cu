// gauss_step.cu -- the Gaussian reverse-diffusion step of the structure (angle) model and the angle wrap that follows it:
// structure_model/sample.py:55-102 (p_sample) + 139-141 (modulo_with_wrapped_range, structure_model/utils.py:20-40).
//
// Reference arithmetic per element (all fp32, every operator rounded separately, in this order):
//   mean = a_t * (x - b_t * out / c_t)            a = 1/sqrt(alpha_t), b = beta_t, c = sqrt(1 - alphabar_t)   sample.py:92-94
//   x'   = t == 0 ? mean : mean + s_t * z         s = sqrt(posterior_variance_t), z ~ N(0,1)                  sample.py:95-101
//   x''  = ((x' - (-pi)) mod 2pi) + (-pi)         torch `%`: fmod, then + 2pi if the remainder is negative     utils.py:33-39
// The per-step scalars come from a host table coef[T,4] = (a, b, c, s) built with the reference's own torch ops.
// z is either handed in (parity runs: "same noise") or drawn in the kernel: Philox4x32-10 keyed by (seed, global graph id,
// 4-element group inside the graph, step) -> Box-Muller, so the stream does not depend on how graphs are sharded over GPUs.
// HBM-bound: 12 B per element (x in, out in, x'' out) + 4 B with explicit noise + 4 B when the per-step history is kept.
#include "common.cuh"
#include "kernels.h"

namespace seqdiff {

constexpr int kGaussThreads = 256;

__device__ __forceinline__ void philox4(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint64_t p0 = static_cast<uint64_t>(0xD2511F53u) * c[0];
    const uint64_t p1 = static_cast<uint64_t>(0xCD9E8D57u) * c[2];
    const uint32_t n0 = static_cast<uint32_t>(p1 >> 32) ^ c[1] ^ k0;
    const uint32_t n1 = static_cast<uint32_t>(p1);
    const uint32_t n2 = static_cast<uint32_t>(p0 >> 32) ^ c[3] ^ k1;
    const uint32_t n3 = static_cast<uint32_t>(p0);
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
// u in (0,1): ((w >> 9) + 0.5) * 2^-23;  (z0, z1) = sqrt(-2 ln u0) * (cos, sin)(2 pi u1)
__device__ __forceinline__ void box_muller(uint32_t w0, uint32_t w1, float& z0, float& z1) {
  const float u0 = (static_cast<float>(w0 >> 9) + 0.5f) * 1.1920928955078125e-07f;
  const float u1 = (static_cast<float>(w1 >> 9) + 0.5f) * 1.1920928955078125e-07f;
  const float r = sqrtf(-2.0f * logf(u0));
  float sn, cs;
  sincospif(2.0f * u1, &sn, &cs);
  z0 = r * cs;
  z1 = r * sn;
}

// the four N(0,1) values of 4-element group q of global graph `graph` at step `step`
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint64_t graph, int q, int step, float (&z)[4]) {
  uint32_t ctr[4] = {static_cast<uint32_t>(q), static_cast<uint32_t>(step), static_cast<uint32_t>(graph), static_cast<uint32_t>(graph >> 32)};
  philox4(ctr, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  box_muller(ctr[0], ctr[1], z[0], z[1]);
  box_muller(ctr[2], ctr[3], z[2], z[3]);
}

// the loop step index from the device counter; with `advance`, the last CTA to have read it moves it on (no separate launch)
__device__ __forceinline__ int loop_step(const int* step_ptr, int* advance) {
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
  return s_sidx;
}

__device__ __forceinline__ float gauss_update(float x, float out, float a, float b, float c, float sd, float z, bool last, bool wrap) {
  const float mean = __fmul_rn(a, __fsub_rn(x, __fdiv_rn(__fmul_rn(b, out), c)));
  const float v = last ? mean : __fadd_rn(mean, __fmul_rn(sd, z));
  return wrap ? wrap_angle(v) : v;  // p_sample alone (sample.py:55-102) returns the un-wrapped value
}

// One thread per group of 4 consecutive elements of one graph (per = L * F elements per graph, groups = ceil(per / 4)).
// PACKED (ragged batch): graph g holds len[g] valid residues of F features, element e of the graph is valid iff e / F < len[g], i.e.
// iff e < len[g] * F.  Valid elements are computed exactly as in the padded kernel, with the Philox counter of their group inside the
// PADDED graph, so they draw the same noise; padded elements are written as 0 without being read, and a group with no valid element
// draws nothing.  With F % 4 != 0 a group can straddle the end of the valid prefix: its valid part is loaded element by element.
template <bool PACKED>
__global__ void __launch_bounds__(kGaussThreads) gauss_step_kernel(const float* __restrict__ coef, int T, int per, const float* x_t,
                                                                   const float* __restrict__ model_out, const float* __restrict__ noise,
                                                                   uint64_t seed, uint64_t graph_id0, int step, const int* __restrict__ step_ptr,
                                                                   float* x_out, float* __restrict__ steps_out,
                                                                   int* __restrict__ advance, int wrap, const uint64_t* __restrict__ rng,
                                                                   const int* __restrict__ len, int F) {
  // x_t / x_out carry no __restrict__: the sampling loop updates the angles in place (each thread reads its 4 elements before it writes them)
  pdl_trigger();
  pdl_wait();
  if (rng) {  // sampling loop: (seed, first global graph id) from device memory -- a cached CUDA graph serves every call
    seed = rng[0];
    graph_id0 = rng[1];
  }
  const size_t n_all = static_cast<size_t>(gridDim.y) * per;
  if (step_ptr) {  // sampling loop: the step index lives on the device; the last CTA to have read it moves it on
    step = loop_step(step_ptr, advance);
    if (noise) noise += static_cast<size_t>(step) * n_all;
  }
  if (step < 0 || step >= T) return;
  const float a = __ldg(coef + 4 * step), b = __ldg(coef + 4 * step + 1), c = __ldg(coef + 4 * step + 2), sd = __ldg(coef + 4 * step + 3);
  const bool last = step == 0;
  if (steps_out) steps_out += static_cast<size_t>(T - 1 - step) * n_all;  // entry k = after the k-th reverse step (sample.py:142-143)
  const int g = blockIdx.y;
  const int groups = (per + 3) >> 2;
  const bool vec = (per & 3) == 0;
  for (int q = blockIdx.x * kGaussThreads + threadIdx.x; q < groups; q += gridDim.x * kGaussThreads) {
    const size_t base = static_cast<size_t>(g) * per + 4 * static_cast<size_t>(q);
    const int cnt = min(4, per - 4 * q);
    int nv = cnt;  // valid elements of the group: a prefix of it
    if constexpr (PACKED) {
      nv = min(cnt, max(0, __ldg(len + g) * F - 4 * q));
      if (nv == 0) {
        if (vec) {
          *reinterpret_cast<float4*>(x_out + base) = make_float4(0.f, 0.f, 0.f, 0.f);
          if (steps_out) *reinterpret_cast<float4*>(steps_out + base) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
          for (int e = 0; e < cnt; ++e) {
            x_out[base + e] = 0.f;
            if (steps_out) steps_out[base + e] = 0.f;
          }
        }
        continue;
      }
    }
    const bool vload = PACKED ? vec && nv == 4 : vec;
    float xv[4], ov[4], zv[4] = {0.f, 0.f, 0.f, 0.f};
    if (vload) {
      const float4 x4 = *reinterpret_cast<const float4*>(x_t + base);
      const float4 o4 = *reinterpret_cast<const float4*>(model_out + base);
      xv[0] = x4.x; xv[1] = x4.y; xv[2] = x4.z; xv[3] = x4.w;
      ov[0] = o4.x; ov[1] = o4.y; ov[2] = o4.z; ov[3] = o4.w;
    } else {
      for (int e = 0; e < 4; ++e) {
        xv[e] = e < nv ? x_t[base + e] : 0.f;
        ov[e] = e < nv ? model_out[base + e] : 0.f;
      }
    }
    if (!last) {
      if (noise) {
        if (vload) {
          const float4 z4 = *reinterpret_cast<const float4*>(noise + base);
          zv[0] = z4.x; zv[1] = z4.y; zv[2] = z4.z; zv[3] = z4.w;
        } else {
          for (int e = 0; e < nv; ++e) zv[e] = noise[base + e];
        }
      } else {
        philox_normal4(seed, graph_id0 + static_cast<uint64_t>(g), q, step, zv);
      }
    }
    float r[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) r[e] = gauss_update(xv[e], ov[e], a, b, c, sd, zv[e], last, wrap != 0);
    if constexpr (PACKED) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (e >= nv) r[e] = 0.f;
    }
    if (vec) {
      const float4 r4 = make_float4(r[0], r[1], r[2], r[3]);
      *reinterpret_cast<float4*>(x_out + base) = r4;
      if (steps_out) *reinterpret_cast<float4*>(steps_out + base) = r4;
    } else {
      for (int e = 0; e < cnt; ++e) {
        x_out[base + e] = r[e];
        if (steps_out) steps_out[base + e] = r[e];
      }
    }
  }
}

int gauss_step(const float* coef, int T, int B, int per_graph, const float* x_t, const float* model_out, const float* noise, uint64_t seed,
               uint64_t graph_id0, int step, const int* step_ptr, float* x_out, float* steps_out, cudaStream_t s, int* advance, bool wrap,
               const uint64_t* rng, const int* len, int F) {
  SD_CHECK(B > 0 && per_graph > 0 && T > 0, "empty Gaussian reverse step");
  SD_CHECK(step_ptr != nullptr || (step >= 0 && step < T), "step index out of range");
  SD_CHECK(!len || (F > 0 && per_graph % F == 0), "packed Gaussian step: per_graph must be a multiple of F");
  const int groups = (per_graph + 3) / 4;
  const dim3 grid(ceil_div(groups, kGaussThreads), B);
  if (len) {
    SD_CUDA(launch_k(gauss_step_kernel<true>, dim3(grid), dim3(kGaussThreads), 0, s, coef, T, per_graph, x_t, model_out, noise, seed, graph_id0, step,
                     step_ptr, x_out, steps_out, advance, wrap ? 1 : 0, rng, len, F));
  } else {
    SD_CUDA(launch_k(gauss_step_kernel<false>, dim3(grid), dim3(kGaussThreads), 0, s, coef, T, per_graph, x_t, model_out, noise, seed, graph_id0, step,
                     step_ptr, x_out, steps_out, advance, wrap ? 1 : 0, rng, static_cast<const int*>(nullptr), 0));
  }
  SD_LAUNCHED("gauss_step", s);
  return SEQDIFF_OK;
}

// ---------------------------------------------------------------------------------------------------
// Backbone score (Model::struct_score): the structure model's training objective at every step k = T-1 .. 0 of a loop.
//   x_k = wrap(sqrt_ac[k] * x0 + sqrt_1m_ac[k] * eps_k)      fp32, __fmul_rn, __fmul_rn, __fadd_rn, wrap_angle (NoisedAnglesDataset)
//   acc += h(wrap(eps_k - pred_k))                           fp64, per element, at the valid positions (angle_loss_terms' arithmetic)
// Both kernels read k from the loop's step counter and (seed, graph_id0) from its RNG words, and take eps_k of element e of graph g
// the way gauss_step_kernel takes its z: from the explicit table noise[k] [B * per], or from Philox at the element's 4-element group
// inside the PADDED graph -- so packed and padded batches draw the same eps at every valid element.  The terms kernel recomputes
// eps_k rather than reading a buffer.  Same thread layout as the Gaussian step: one thread per group of 4 consecutive elements.
__device__ __forceinline__ void step_noise4(const float* noise, size_t base, int nv, bool vload, uint64_t seed, uint64_t graph, int q, int step,
                                            float (&z)[4]) {
  if (noise) {
    if (vload) {
      const float4 z4 = *reinterpret_cast<const float4*>(noise + base);
      z[0] = z4.x; z[1] = z4.y; z[2] = z4.z; z[3] = z4.w;
    } else {
      for (int e = 0; e < nv; ++e) z[e] = noise[base + e];
    }
  } else {
    philox_normal4(seed, graph, q, step, z);
  }
}

// x_t [B, per]: padded -> every element; PACKED -> the valid elements (e < len[g] * F), padded ones are neither read nor written.
template <bool PACKED>
__global__ void __launch_bounds__(kGaussThreads) angle_qsample_kernel(const float* __restrict__ qs, int per, const float* __restrict__ x0,
                                                                      const float* __restrict__ noise, const int* __restrict__ step_ptr,
                                                                      const uint64_t* __restrict__ rng, const int* __restrict__ len, int F,
                                                                      float* __restrict__ x_t) {
  pdl_trigger();
  pdl_wait();
  const int step = loop_step(step_ptr, nullptr);
  const uint64_t seed = rng[0], graph_id0 = rng[1];
  const int g = blockIdx.y;
  if (noise) noise += static_cast<size_t>(step) * gridDim.y * per;
  const float sa = __ldg(qs + 2 * step), sb = __ldg(qs + 2 * step + 1);
  const int groups = (per + 3) >> 2;
  const bool vec = (per & 3) == 0;
  for (int q = blockIdx.x * kGaussThreads + threadIdx.x; q < groups; q += gridDim.x * kGaussThreads) {
    const size_t base = static_cast<size_t>(g) * per + 4 * static_cast<size_t>(q);
    int nv = min(4, per - 4 * q);
    if constexpr (PACKED) {
      nv = min(nv, max(0, __ldg(len + g) * F - 4 * q));
      if (nv == 0) continue;
    }
    const bool vload = vec && nv == 4;
    float xv[4] = {0.f, 0.f, 0.f, 0.f}, zv[4] = {0.f, 0.f, 0.f, 0.f};
    if (vload) {
      const float4 x4 = *reinterpret_cast<const float4*>(x0 + base);
      xv[0] = x4.x; xv[1] = x4.y; xv[2] = x4.z; xv[3] = x4.w;
    } else {
      for (int e = 0; e < nv; ++e) xv[e] = x0[base + e];
    }
    step_noise4(noise, base, nv, vload, seed, graph_id0 + static_cast<uint64_t>(g), q, step, zv);
    float r[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) r[e] = wrap_angle(__fadd_rn(__fmul_rn(sa, xv[e]), __fmul_rn(sb, zv[e])));
    if (vload) {
      *reinterpret_cast<float4*>(x_t + base) = make_float4(r[0], r[1], r[2], r[3]);
    } else {
      for (int e = 0; e < nv; ++e) x_t[base + e] = r[e];
    }
  }
}

// acc [B, per] fp64 += h(wrap(eps - pred)) at the valid elements: padded -> mask[g * (per / F) + e / F] != 0, PACKED -> e < len[g] * F.
// Every element is owned by one thread and summed in step order (no atomics): bit-reproducible.  Other elements are never read or
// written.  The last CTA to have read the step counter moves it on.
template <bool PACKED>
__global__ void __launch_bounds__(kGaussThreads) angle_score_terms_kernel(int per, const float* __restrict__ pred, const float* __restrict__ noise,
                                                                          const float* __restrict__ mask, const int* __restrict__ step_ptr,
                                                                          int* __restrict__ advance, const uint64_t* __restrict__ rng,
                                                                          const int* __restrict__ len, int F, double* __restrict__ acc) {
  pdl_trigger();
  pdl_wait();
  const int step = loop_step(step_ptr, advance);
  const uint64_t seed = rng[0], graph_id0 = rng[1];
  const int g = blockIdx.y;
  if (noise) noise += static_cast<size_t>(step) * gridDim.y * per;
  const int groups = (per + 3) >> 2;
  const bool vec = (per & 3) == 0;
  for (int q = blockIdx.x * kGaussThreads + threadIdx.x; q < groups; q += gridDim.x * kGaussThreads) {
    const size_t base = static_cast<size_t>(g) * per + 4 * static_cast<size_t>(q);
    const int cnt = min(4, per - 4 * q);
    bool valid[4] = {false, false, false, false};
    int nv = 0;  // packed: valid elements form a prefix of the group
    if constexpr (PACKED) {
      nv = min(cnt, max(0, __ldg(len + g) * F - 4 * q));
      for (int e = 0; e < 4; ++e) valid[e] = e < nv;
    } else {
      for (int e = 0; e < cnt; ++e) {
        valid[e] = __ldg(mask + static_cast<size_t>(g) * (per / F) + (4 * q + e) / F) != 0.f;
        nv += valid[e] ? 1 : 0;
      }
    }
    if (nv == 0) continue;
    const bool vload = vec && nv == 4;
    float zv[4] = {0.f, 0.f, 0.f, 0.f};
    // explicit noise: element-wise loads cover the valid ones only (padded mode may have holes, so nv is not a prefix length there)
    if (noise && !vload) {
      for (int e = 0; e < 4; ++e)
        if (valid[e]) zv[e] = noise[base + e];
    } else {
      step_noise4(noise, base, 4, vload, seed, graph_id0 + static_cast<uint64_t>(g), q, step, zv);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (valid[e]) acc[base + e] += static_cast<double>(angle_smooth_l1(wrap_angle(__fsub_rn(zv[e], pred[base + e]))));
  }
}

int angle_qsample(const float* qs, int B, int per_graph, const float* x0, const float* noise, const int* step_ptr, const uint64_t* rng,
                  float* x_t, cudaStream_t s, const int* len, int F) {
  SD_CHECK(B > 0 && per_graph > 0 && F > 0 && per_graph % F == 0, "angle q-sample: per_graph must be a positive multiple of F");
  SD_CHECK(step_ptr && rng, "angle q-sample runs inside a loop (step counter and RNG words on the device)");
  const dim3 grid(ceil_div((per_graph + 3) / 4, kGaussThreads), B);
  if (len) {
    SD_CUDA(launch_k(angle_qsample_kernel<true>, grid, dim3(kGaussThreads), 0, s, qs, per_graph, x0, noise, step_ptr, rng, len, F, x_t));
  } else {
    SD_CUDA(launch_k(angle_qsample_kernel<false>, grid, dim3(kGaussThreads), 0, s, qs, per_graph, x0, noise, step_ptr, rng,
                     static_cast<const int*>(nullptr), F, x_t));
  }
  SD_LAUNCHED("angle_qsample", s);
  return SEQDIFF_OK;
}

int angle_score_terms(int B, int per_graph, const float* pred, const float* noise, const float* mask, const int* step_ptr, int* advance,
                      const uint64_t* rng, double* acc, cudaStream_t s, const int* len, int F) {
  SD_CHECK(B > 0 && per_graph > 0 && F > 0 && per_graph % F == 0, "angle score terms: per_graph must be a positive multiple of F");
  SD_CHECK(step_ptr && advance && rng, "angle score terms run inside a loop (step counter and RNG words on the device)");
  const dim3 grid(ceil_div((per_graph + 3) / 4, kGaussThreads), B);
  if (len) {
    SD_CUDA(launch_k(angle_score_terms_kernel<true>, grid, dim3(kGaussThreads), 0, s, per_graph, pred, noise, mask, step_ptr, advance, rng, len,
                     F, acc));
  } else {
    SD_CUDA(launch_k(angle_score_terms_kernel<false>, grid, dim3(kGaussThreads), 0, s, per_graph, pred, noise, mask, step_ptr, advance, rng,
                     static_cast<const int*>(nullptr), F, acc));
  }
  SD_LAUNCHED("angle_score_terms", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
