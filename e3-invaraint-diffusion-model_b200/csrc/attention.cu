// attention.cu -- the 15 attention cores per forward (3 SELayer + 6 self + 6 cross), i.e. HF
// BertSelfAttention with transformers-4.38.2 `relative_key` semantics (SURVEY.md Appendix A):
//
//   S[l,r]  = ( q_l . k_r  +  q_l . E[l - r + P - 1] ) / 8  +  (1 - mask[r]) * -10000
//   out_l   = softmax_r(S[l,:]) @ V
//
// E = distance_embedding [2P-1, 64], shared by all heads; cross-attention has no E term.
//
// 16-bit modes (bf16 or fp16 operands): the persistent pipelined tcgen05 kernel of attention_pipe.cu, for every shape.
// fp32 kernel (parity mode): one warp per query row, straight loops.
#include "common.cuh"
#include "kernels.h"

namespace seqdiff {

template <>
int attention<bf16>(int B, int heads, int Lq, int Lk, const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv,
                    const bf16* dist_emb, int P, const float* key_mask, bf16* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
  return attention_pipe<bf16>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, kv_div);
}
template <>
int attention<f16>(int B, int heads, int Lq, int Lk, const f16* q, int ldq, const f16* k, int ldk, const f16* v, int ldv,
                   const f16* dist_emb, int P, const float* key_mask, f16* out, cudaStream_t s, const AttnPack* pack, int kv_div) {
  return attention_pipe<f16>(B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, dist_emb, P, key_mask, out, s, pack, kv_div);
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
