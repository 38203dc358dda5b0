// decode_loss.cu -- the two per-residue reductions that follow the denoiser in the reference:
//   decode_sequences : the per-graph loop at the end of denoise(), sequence_model/sample.py:208-224 (argmax decode of the final
//                      tensor and of the true sequence, recovery rate over the masked positions);
//   loss_terms       : the reductions of PeptideDiff.get_loss (sequence_model/model.py:313-345) and elbo_loss
//                      (sequence_model/utils.py:132-161).
// Both are HBM-bound streams over [N,20] fp32 rows (80 B per row and per input tensor); integer outputs are exact, the
// floating-point sums are accumulated in fp64 with a fixed reduction order (deterministic run to run).
#include "common.cuh"
#include "kernels.h"

namespace seqdiff {

constexpr int C = SEQDIFF_NUM_CLASSES;
constexpr int kDecThreads = 128;

__device__ __forceinline__ void load_row20(const float* __restrict__ p, float (&r)[C]) {
#pragma unroll
  for (int j4 = 0; j4 < C; j4 += 4) {
    const float4 a = *reinterpret_cast<const float4*>(p + j4);
    r[j4] = a.x; r[j4 + 1] = a.y; r[j4 + 2] = a.z; r[j4 + 3] = a.w;
  }
}
// first maximum wins (torch.argmax); NaN never compares greater, as in the reverse step
__device__ __forceinline__ int argmax20(const float (&r)[C]) {
  int best = 0;
  float bv = r[0];
#pragma unroll
  for (int j = 1; j < C; ++j)
    if (r[j] > bv) { bv = r[j]; best = j; }
  return best;
}

// one CTA per graph
__global__ void __launch_bounds__(kDecThreads) decode_kernel(int L, const float* __restrict__ fin, const float* __restrict__ tru,
                                                             const float* __restrict__ mask, uint8_t* __restrict__ pred_idx,
                                                             uint8_t* __restrict__ true_idx, int* __restrict__ counts) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x;
  int hit = 0, valid = 0;
  for (int l = threadIdx.x; l < L; l += kDecThreads) {
    const size_t n = static_cast<size_t>(b) * L + l;
    float r[C];
    load_row20(fin + n * C, r);
    const int p = argmax20(r);
    load_row20(tru + n * C, r);
    const int t = argmax20(r);
    pred_idx[n] = static_cast<uint8_t>(p);
    true_idx[n] = static_cast<uint8_t>(t);
    const bool m = mask[n] != 0.f;  // ligand_mask[i].bool()
    valid += m ? 1 : 0;
    hit += (m && p == t) ? 1 : 0;
  }
  __shared__ int s_hit[kDecThreads / 32], s_valid[kDecThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    hit += __shfl_xor_sync(0xffffffffu, hit, o);
    valid += __shfl_xor_sync(0xffffffffu, valid, o);
  }
  if ((threadIdx.x & 31) == 0) { s_hit[threadIdx.x >> 5] = hit; s_valid[threadIdx.x >> 5] = valid; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int h = 0, v = 0;
    for (int w = 0; w < kDecThreads / 32; ++w) { h += s_hit[w]; v += s_valid[w]; }
    counts[2 * b] = h;
    counts[2 * b + 1] = v;
  }
}

int decode_sequences(int B, int L, const float* final_seq, const float* true_seq, const float* mask, uint8_t* pred_idx, uint8_t* true_idx,
                     int* counts, cudaStream_t s) {
  SD_CHECK(B > 0 && L > 0, "empty decode");
  SD_CUDA(launch_k(decode_kernel, dim3(B), dim3(kDecThreads), 0, s, L, final_seq, true_seq, mask, pred_idx, true_idx, counts));
  SD_LAUNCHED("decode", s);
  return SEQDIFF_OK;
}

// ---------------------------------------------------------------------------------------------------
constexpr int kLossThreads = 256;
constexpr int kLossTerms = 10;
constexpr int kLossMaxCtas = 296;

// log-sum-exp of a row in fp32 the way torch's log_softmax does it: max, sum of expf(x - max), logf
__device__ __forceinline__ float lse20(const float (&r)[C], float& mx) {
  mx = r[0];
#pragma unroll
  for (int j = 1; j < C; ++j) mx = fmaxf(mx, r[j]);
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) sum += expf(r[j] - mx);
  return logf(sum);
}

__global__ void __launch_bounds__(kLossThreads) loss_terms_kernel(int N, const float* __restrict__ logits, const float* __restrict__ x0,
                                                                  const float* __restrict__ x_t, const float* __restrict__ mask,
                                                                  double* __restrict__ partial, unsigned* __restrict__ arrive,
                                                                  double* __restrict__ terms) {
  pdl_trigger();
  pdl_wait();
  double acc[kLossTerms];
#pragma unroll
  for (int k = 0; k < kLossTerms; ++k) acc[k] = 0.0;
  for (int n = blockIdx.x * kLossThreads + threadIdx.x; n < N; n += gridDim.x * kLossThreads) {
    float lg[C], r[C];
    load_row20(x0 + static_cast<size_t>(n) * C, r);
    const int tgt = argmax20(r);
    // q = softmax(x0 row) (utils.py:147); F.kl_div takes log q from q itself (xlogy), not from log_probs2 (utils.py:152 is unused)
    float q[C];
    {
      float mx0 = r[0];
#pragma unroll
      for (int j = 1; j < C; ++j) mx0 = fmaxf(mx0, r[j]);
      float sum0 = 0.f;
#pragma unroll
      for (int j = 0; j < C; ++j) { q[j] = expf(r[j] - mx0); sum0 += q[j]; }
#pragma unroll
      for (int j = 0; j < C; ++j) q[j] = __fdiv_rn(q[j], sum0);
    }
    load_row20(x_t + static_cast<size_t>(n) * C, r);
    const int xt = argmax20(r);
    load_row20(logits + static_cast<size_t>(n) * C, lg);
    const int pred = argmax20(lg);
    const bool m = mask[n] != 0.f;
    const bool noised = xt != tgt;
    const bool sel = m && !noised;
    acc[0] += m ? 1.0 : 0.0;
    acc[1] += noised ? 1.0 : 0.0;
    acc[2] += sel ? 1.0 : 0.0;
    acc[3] += (m && xt == tgt) ? 1.0 : 0.0;
    acc[4] += (m && pred == tgt) ? 1.0 : 0.0;
    if (noised || sel) {
      float mx;
      const float lse = lse20(lg, mx);
      const float ce = -(lg[tgt] - mx - lse);  // CrossEntropyLoss row term: -log_softmax(logits)[target]
      if (noised) acc[5] += ce;
      if (sel) acc[6] += ce;
      if (noised) {
        float le[C], mxe;
#pragma unroll
        for (int j = 0; j < C; ++j) le[j] = lg[j] + 1e-6f;
        const float lsee = lse20(le, mxe);
        float ent = 0.f, kl = 0.f;
#pragma unroll
        for (int j = 0; j < C; ++j) {
          const float lp = le[j] - mxe - lsee;               // log_softmax(logits + eps)
          const float p = expf(lg[j] - mx - lse);            // softmax(logits)
          ent += p * lp;
          kl += q[j] * logf(q[j]) - q[j] * lp;               // F.kl_div(log_probs1, probs2): xlogy(q, q) - q * log_probs1
        }
        acc[7] += ent;
        acc[8] += kl;
      }
    }
  }
  // block reduction in a fixed order, then the last CTA to arrive folds the per-CTA partials in CTA order
  __shared__ double s_acc[kLossThreads / 32][kLossTerms];
#pragma unroll
  for (int k = 0; k < kLossTerms; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_acc[threadIdx.x >> 5][k] = v;
  }
  __syncthreads();
  __shared__ bool s_last;
  if (threadIdx.x < kLossTerms) {
    double v = 0.0;
    for (int w = 0; w < kLossThreads / 32; ++w) v += s_acc[w][threadIdx.x];
    partial[static_cast<size_t>(blockIdx.x) * kLossTerms + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(arrive, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    __threadfence();
    if (threadIdx.x < kLossTerms) {
      double v = 0.0;
      for (unsigned c = 0; c < gridDim.x; ++c) v += reinterpret_cast<const volatile double*>(partial)[static_cast<size_t>(c) * kLossTerms + threadIdx.x];
      terms[threadIdx.x] = v;
    }
    if (threadIdx.x == 0) *arrive = 0u;
  }
}

size_t loss_terms_scratch_bytes() { return (static_cast<size_t>(kLossMaxCtas) * kLossTerms + 2) * sizeof(double); }
// per-CTA partials + arrival counter.  The training steps hand in scratch from their own workspace: a cudaMallocAsync per optimizer
// step can stall the launching thread for milliseconds whenever the pool has been trimmed at a synchronisation (seen as 3 - 90 ms
// gaps in front of this launch in the per-kernel profiles of the training step).  The stand-alone entry points keep stream-ordered
// scratch, so concurrent calls on different streams never share it, with the pool told to keep what it has instead of returning it
// to the OS at every synchronisation.
static cudaError_t stream_scratch(double** out, size_t bytes, cudaStream_t s) {
  static const bool pool_kept = [] {
    int dev = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      uint64_t keep = 64ull << 20;  // bytes the pool may hold across synchronisations (this scratch is 24 KB)
      uint64_t cur = 0;
      if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &cur) == cudaSuccess && cur < keep)
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
    return true;
  }();
  (void)pool_kept;
  return cudaMallocAsync(reinterpret_cast<void**>(out), bytes, s);
}
int loss_terms(int N, const float* logits, const float* x0, const float* x_t, const float* mask, double* terms, cudaStream_t s, double* scratch_in) {
  SD_CHECK(N > 0, "empty loss");
  int ctas = ceil_div(N, kLossThreads);
  if (ctas > kLossMaxCtas) ctas = kLossMaxCtas;
  const size_t bytes = (static_cast<size_t>(ctas) * kLossTerms + 2) * sizeof(double);
  double* scratch = scratch_in;
  if (!scratch) SD_CUDA(stream_scratch(&scratch, bytes, s));
  unsigned* arrive = reinterpret_cast<unsigned*>(scratch + static_cast<size_t>(ctas) * kLossTerms);
  cudaError_t e = cudaMemsetAsync(arrive, 0, 2 * sizeof(double), s);
  if (e == cudaSuccess) e = launch_k(loss_terms_kernel, dim3(ctas), dim3(kLossThreads), 0, s, N, logits, x0, x_t, mask, scratch, arrive, terms);
  const cudaError_t ef = scratch_in ? cudaSuccess : cudaFreeAsync(scratch, s);
  SD_CUDA(e);
  SD_CUDA(ef);
  SD_LAUNCHED("loss_terms", s);
  return SEQDIFF_OK;
}

// ---------------------------------------------------------------------------------------------------
// Objective of the structure (angle) model: wrapped smooth-L1 on the predicted noise, per feature, over the valid ligand positions.
//   d = wrap(known_noise - pred) into [-pi, pi);  h(d) = 0.5 d^2 / beta (|d| < beta), |d| - 0.5 beta otherwise;  beta = pi / 10.
// terms[i] = sum of h over the valid positions of feature i (i < F), terms[F] = number of valid positions; loss = mean_i terms[i] / terms[F].
// wrap_angle and h (angle_smooth_l1) are common.cuh's, shared with the sampler and the backbone score.

template <int F>
__global__ void __launch_bounds__(kLossThreads) angle_loss_terms_kernel(int N, const float* __restrict__ pred, const float* __restrict__ noise,
                                                                        const float* __restrict__ mask, double* __restrict__ partial,
                                                                        unsigned* __restrict__ arrive, double* __restrict__ terms) {
  pdl_trigger();
  pdl_wait();
  constexpr int NT = F + 1;
  double acc[NT];
#pragma unroll
  for (int k = 0; k < NT; ++k) acc[k] = 0.0;
  for (int n = blockIdx.x * kLossThreads + threadIdx.x; n < N; n += gridDim.x * kLossThreads) {
    if (mask[n] == 0.f) continue;
    acc[F] += 1.0;
#pragma unroll
    for (int i = 0; i < F; ++i) {
      const size_t e = static_cast<size_t>(n) * F + i;
      acc[i] += angle_smooth_l1(wrap_angle(__fsub_rn(noise[e], pred[e])));
    }
  }
  // fixed-order reduction (deterministic run to run): warp shuffles, warps in order, then the last CTA folds the partials in CTA order
  __shared__ double s_acc[kLossThreads / 32][NT];
#pragma unroll
  for (int k = 0; k < NT; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_acc[threadIdx.x >> 5][k] = v;
  }
  __syncthreads();
  __shared__ bool s_last;
  if (threadIdx.x < NT) {
    double v = 0.0;
    for (int w = 0; w < kLossThreads / 32; ++w) v += s_acc[w][threadIdx.x];
    partial[static_cast<size_t>(blockIdx.x) * NT + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(arrive, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    __threadfence();
    if (threadIdx.x < NT) {
      double v = 0.0;
      for (unsigned c = 0; c < gridDim.x; ++c) v += reinterpret_cast<const volatile double*>(partial)[static_cast<size_t>(c) * NT + threadIdx.x];
      terms[threadIdx.x] = v;
    }
    if (threadIdx.x == 0) *arrive = 0u;
  }
}

// dL/dpred = -h'(d) / (F * n_valid) at valid positions, 0 elsewhere; h'(d) = d / beta or sign(d).  n_valid = terms[F], read on the
// device (no host synchronisation); a batch without a valid position (n_valid = 0) gets a zero gradient.
template <int F>
__global__ void __launch_bounds__(256) angle_loss_bwd_kernel(int N, const float* __restrict__ pred, const float* __restrict__ noise,
                                                             const float* __restrict__ mask, const double* __restrict__ terms,
                                                             float* __restrict__ dpred) {
  pdl_wait();
  const double n_valid = terms[F];
  const float scale = n_valid > 0.0 ? static_cast<float>(-1.0 / (static_cast<double>(F) * n_valid)) : 0.f;
  for (int e = blockIdx.x * 256 + threadIdx.x; e < N * F; e += gridDim.x * 256) {
    float g = 0.f;
    if (mask[e / F] != 0.f) {
      const float d = wrap_angle(__fsub_rn(noise[e], pred[e]));
      g = scale * (fabsf(d) < kAngleBeta ? d / kAngleBeta : (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)));
    }
    dpred[e] = g;
  }
}

size_t angle_loss_scratch_bytes() { return (static_cast<size_t>(kLossMaxCtas) * (kAngleMaxF + 1) + 2) * sizeof(double); }
int angle_loss_terms(int N, int F, const float* pred, const float* noise, const float* mask, double* terms, cudaStream_t s, double* scratch_in) {
  SD_CHECK(N > 0, "empty loss");
  SD_CHECK(F == 8 || F == 20, "angle loss: feature_size must be 8 or 20");
  int ctas = ceil_div(N, kLossThreads);
  if (ctas > kLossMaxCtas) ctas = kLossMaxCtas;
  const size_t bytes = (static_cast<size_t>(ctas) * (F + 1) + 2) * sizeof(double);
  double* scratch = scratch_in;
  if (!scratch) SD_CUDA(stream_scratch(&scratch, bytes, s));
  unsigned* arrive = reinterpret_cast<unsigned*>(scratch + static_cast<size_t>(ctas) * (F + 1));
  cudaError_t e = cudaMemsetAsync(arrive, 0, 2 * sizeof(double), s);
  if (e == cudaSuccess) {
    if (F == 8) e = launch_k(angle_loss_terms_kernel<8>, dim3(ctas), dim3(kLossThreads), 0, s, N, pred, noise, mask, scratch, arrive, terms);
    else e = launch_k(angle_loss_terms_kernel<20>, dim3(ctas), dim3(kLossThreads), 0, s, N, pred, noise, mask, scratch, arrive, terms);
  }
  const cudaError_t ef = scratch_in ? cudaSuccess : cudaFreeAsync(scratch, s);
  SD_CUDA(e);
  SD_CUDA(ef);
  SD_LAUNCHED("angle_loss_terms", s);
  return SEQDIFF_OK;
}
int angle_loss_bwd(int N, int F, const float* pred, const float* noise, const float* mask, const double* terms, float* dpred, cudaStream_t s) {
  SD_CHECK(N > 0, "empty loss");
  SD_CHECK(F == 8 || F == 20, "angle loss: feature_size must be 8 or 20");
  const int grid = ceil_div(N * F, 256);
  if (F == 8) SD_CUDA(launch_k(angle_loss_bwd_kernel<8>, dim3(grid), dim3(256), 0, s, N, pred, noise, mask, terms, dpred));
  else SD_CUDA(launch_k(angle_loss_bwd_kernel<20>, dim3(grid), dim3(256), 0, s, N, pred, noise, mask, terms, dpred));
  SD_LAUNCHED("angle_loss_bwd", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
