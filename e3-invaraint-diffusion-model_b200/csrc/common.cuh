// common.cuh -- shared helpers for the seqdiff sm_100a kernels: error plumbing, launch counting,
// bf16 conversion, and the inline-PTX wrappers for mbarrier / TMA / tcgen05 (Blackwell only).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>

#include "../../include/seqdiff_b200.h"

namespace seqdiff {

// ---- error handling ------------------------------------------------------------------------------
void set_error(const std::string& msg);
extern std::atomic<uint64_t> g_launches;

#define SD_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      ::seqdiff::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                           std::to_string(__LINE__));                                              \
      return SEQDIFF_ERR_CUDA;                                                                     \
    }                                                                                              \
  } while (0)

#define SD_CHECK(cond, msg)                                                                        \
  do {                                                                                             \
    if (!(cond)) {                                                                                 \
      ::seqdiff::set_error(std::string(msg) + " [" #cond "] @" + __FILE__ + ":" + std::to_string(__LINE__)); \
      return SEQDIFF_ERR_INVALID;                                                                  \
    }                                                                                              \
  } while (0)

#define SD_TRY(expr)                  \
  do {                                \
    int _r = (expr);                  \
    if (_r != SEQDIFF_OK) return _r;  \
  } while (0)

// every kernel launch goes through this so `gpu_launches` in bench.py is a count, not a guess; with the
// event profiler on (seqdiff_profile_begin) it also drops a CUDA event behind the kernel on its stream.
void profile_mark(const char* tag, cudaStream_t s);
extern bool g_profiling;
#define SD_LAUNCHED(tag, stream)                                   \
  do {                                                             \
    ::seqdiff::g_launches.fetch_add(1, std::memory_order_relaxed); \
    SD_CUDA(cudaGetLastError());                                   \
    if (::seqdiff::g_profiling) ::seqdiff::profile_mark(tag, stream); \
  } while (0)

typedef __nv_bfloat16 bf16;
typedef __half f16;

// ---- element conversion --------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<f16>(f16 v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }
// fp16 conversions saturate to +-65504 instead of producing inf (the fp16 mode's only range hazard)
__device__ __forceinline__ float sat_f16(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
template <> __device__ __forceinline__ f16 from_f32<f16>(float v) { return __float2half_rn(sat_f16(v)); }

// 8 consecutive elements <-> 8 floats (16B for bf16, 32B for f32); pointers must be 16B aligned
template <typename T> __device__ __forceinline__ void load8(const T* p, float (&v)[8]);
template <> __device__ __forceinline__ void load8<float>(const float* p, float (&v)[8]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <> __device__ __forceinline__ void load8<bf16>(const bf16* p, float (&v)[8]) {
  uint4 r = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 t = __floats2half2_rn(sat_f16(lo), sat_f16(hi));
  return *reinterpret_cast<uint32_t*>(&t);
}
// two floats -> one 32-bit word of the 16-bit operand type T
template <typename T> __device__ __forceinline__ uint32_t pack2(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2<bf16>(float lo, float hi) { return pack_bf16x2(lo, hi); }
template <> __device__ __forceinline__ uint32_t pack2<f16>(float lo, float hi) { return pack_f16x2(lo, hi); }
template <> __device__ __forceinline__ void load8<f16>(const f16* p, float (&v)[8]) {
  uint4 r = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
template <typename T> __device__ __forceinline__ void store8(T* p, const float (&v)[8]);
template <> __device__ __forceinline__ void store8<float>(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void store8<bf16>(bf16* p, const float (&v)[8]) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]); r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]); r.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

template <> __device__ __forceinline__ void store8<f16>(f16* p, const float (&v)[8]) {
  uint4 r;
  r.x = pack_f16x2(v[0], v[1]); r.y = pack_f16x2(v[2], v[3]);
  r.z = pack_f16x2(v[4], v[5]); r.w = pack_f16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = r;
}

// exact-erf GELU (nn.GELU() / HF "gelu": model.py:43,133) and SiLU
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// 16-bit-mode GELU for the tcgen05 GEMM epilogue.  erf by Abramowitz-Stegun 7.1.25 (|err| <= 2.5e-5, an order of
// magnitude below fp16 output resolution), folded so one element costs ~11 issue slots (2 of them MUFU):
//   gelu(x) = max(x,0) - 0.5|x| (a1 t + a2 t^2 + a3 t^3) exp(-x^2/2),   t = 1 / (1 + p |x| / sqrt2)
// (the libdevice erff path costs ~35 and made the epilogue, not the MMA, the bound of the GELU GEMMs).
__device__ __forceinline__ float gelu_fast(float x) {
  const float ax = fabsf(x);
  const float t = rcp_approx(fmaf(ax, 0.33267254f, 1.0f));
  const float poly = t * fmaf(t, fmaf(t, 0.3739278f, -0.0479399f), 0.1740121f);  // a_i / 2
  const float e = ex2_approx(x * x * -0.72134752f);                              // exp(-x^2/2)
  return fmaf(-ax * poly, e, fmaxf(x, 0.0f));
}
__device__ __forceinline__ float silu(float x) { return x / (1.0f + expf(-x)); }
__device__ __forceinline__ float silu_fast(float x) { return x * rcp_approx(1.0f + ex2_approx(x * -1.44269504f)); }

// ---- PTX: shared-memory addresses, mbarrier ----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  uint32_t spins = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    // watchdog: a lost TMA / MMA completion must fault the launch, never hang the GPU
    if (!done && ++spins > (1u << 24)) __trap();
  } while (!done);
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- PTX: TMA (cp.async.bulk.tensor) --------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load global -> shared, completion signalled on `bar` (complete_tx::bytes)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// 3-D tile store shared -> global (bulk async group); rows / columns outside the tensor are clipped
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// 2-D tile store shared -> global (bulk async group); rows / columns outside the tensor are clipped
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// at most one bulk store of this thread may still be reading its smem source
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all bulk stores of this thread have finished READING their smem source (the tile may be overwritten)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... and have fully completed (writes visible) -- required before the kernel exits / signals dependents
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- PTX: tcgen05 / TMEM ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread for the whole CTA
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on `bar` once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- PTX: CTA pairs (cta_group::2) -- one tcgen05.mma spans the two SMs of a cluster of 2 -------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA tile load into THIS CTA's smem whose completion is signalled on a barrier that may live in the peer CTA
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 from each CTA's smem] * B[N: N/2 from each CTA's smem]; issued by the leader CTA only
__device__ __forceinline__ void umma_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior MMAs of this thread completed) on the barrier at this smem offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ---- warp-uniform single-issuer variants ---------------------------------------------------------------------
// tcgen05.mma / tcgen05.commit / cp.async.bulk.tensor are issued once per WARP on the uniform datapath.  Inside an
// `if (lane == 0)` region ptxas must assume divergent operands and wraps every such instruction in an ELECT + 5x R2UR
// waterfall loop (~100 cycles per MMA: measured as the issue bound of every kernel here).  Called from warp-convergent
// code instead -- the whole warp runs the role loop, operands derive from uniform values (blockIdx, loop counters, a
// __shfl-broadcast warp index) -- these compile to back-to-back UTCHMMA / UTCBAR / UTMALDG with descriptors in uniform
// registers.  elect.sync picks the issuing lane (the same lane every time for a full mask).
__device__ __forceinline__ int warp_id_uniform() { return __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0); }
__device__ __forceinline__ void umma_bf16_e(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_cg2_e(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_e(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc_e(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
      "h"(mask)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_e(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
      "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_e(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_cg2_e(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}

// UMMA shared-memory matrix descriptor, K-major operand tile [rows][64 bf16] written by TMA with
// SWIZZLE_128B: 8-row x 128B swizzle atoms, 1024B apart (SBO); LBO unused for swizzled K-major.
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address  [0,14)
  d |= static_cast<uint64_t>(1) << 16;                       // LBO (16B units) [16,30)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;               // SBO            [32,46)
  d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                       // SWIZZLE_128B
  return d;
}
// MN-major operand, SWIZZLE_128B: the tile is stored as [k][mn] with 64 mn-elements (128 B) per k-row -- what a TMA box of
// 64 rows x 64 columns of a row-major [k, mn] matrix leaves in shared memory.  Canonical layout (cute: ((8,n),(8,k)):((1,LBO),(8,SBO))
// in 16 B units): 8 k-rows of 128 B form a 1 KB swizzle group, SBO = stride between groups along k (1024 B), LBO = stride between
// 64-element blocks along mn (`mn_block_stride`, the size of one TMA box).  A k-step of 16 advances the start address by 2048 B.
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t mn_block_stride) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((mn_block_stride >> 4) & 0x3FFFu) << 16;  // LBO
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                           // SBO
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
constexpr uint32_t kUmmaAMnMajor = 1u << 15, kUmmaBMnMajor = 1u << 16;  // instruction-descriptor bits: operand is MN-major
// instruction descriptor, kind::f16: {f16|bf16} x {f16|bf16} -> f32, both operands K-major.
// a_fmt / b_fmt: 0 = F16, 1 = BF16 (cute::UMMA::F16F32Format)
__host__ __device__ constexpr uint32_t umma_idesc_16(int M, int N, uint32_t a_fmt, uint32_t b_fmt) {
  return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// ---- SEQDIFF_DEBUG_BOUNDS build (python build.py with SEQDIFF_DEBUG_BOUNDS=1 -> libseqdiff_b200_dbg.so) --------------------------
// The GPU pool does not allow compute-sanitizer, so the debug build carries its own checks:
//  * SD_DEV_ASSERT(cond): device-side assert (printf + trap) on indices taken from device-resident maps and counters;
//  * guard bands: every buffer carved out of a workspace (Bump in model.cu, Arena in train.cu) is followed by 256 B filled with a
//    pattern by a kernel on the launching stream; seqdiff_debug_check_guards() verifies all of them -- an out-of-bounds write past
//    the end of any activation / tape buffer shows up as a broken band.  In the product build all of this compiles to nothing.
#ifdef SEQDIFF_DEBUG_BOUNDS
#define SD_DEV_ASSERT(cond)                                                                                              \
  do {                                                                                                                   \
    if (!(cond)) {                                                                                                       \
      printf("SD_DEV_ASSERT failed: %s at %s:%d (block %d,%d thread %d)\n", #cond, __FILE__, __LINE__, blockIdx.x, blockIdx.y, threadIdx.x); \
      __trap();                                                                                                          \
    }                                                                                                                    \
  } while (0)
constexpr size_t kGuardBytes = 256;
#else
#define SD_DEV_ASSERT(cond) ((void)0)
constexpr size_t kGuardBytes = 0;
#endif
// (debug build) registers + fills the guard band at `p`; `owner` groups the bands of one workspace carve (re-carving replaces them)
int debug_guard_begin(const void* owner);
int debug_guard_add(const void* owner, void* p, cudaStream_t s);
int debug_guard_check(cudaStream_t s, int* n_bands, int* n_broken);

// ---- programmatic dependent launch (PDL) ----------------------------------------------------------------
// Every kernel of the path is launched with cudaLaunchAttributeProgrammaticStreamSerialization: it may become resident
// while its predecessor drains, runs its prologue (smem carve-up, mbarrier init, TMEM alloc, descriptor prefetch), and then
// blocks in pdl_wait() until the predecessor grid has completed and flushed -- before its first dependent global access.
// pdl_trigger() lets the successor start being scheduled.  Both are no-ops without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
int pdl_scope_exchange(int mode);  // sets the calling thread's scope mode (0 = none), returns the previous one
int pdl_mode();  // effective mode of this launch: 0 off, 1 every launch, 3 only heavy successors (>= 64 KB of shared memory)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kc(int cluster_x, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int n = 0;
  const int pm = pdl_mode();  // 0 off | 1 every launch | 3 heavy successors only (model.cu)
  if (pm == 1 || (pm == 3 && smem >= 65536)) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = static_cast<unsigned>(cluster_x);
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  return launch_kc(1, kernel, grid, block, smem, s, args...);
}

// ---- angles of the structure model: one definition for the sampler, the training loss and the backbone score --------------------
// modulo_with_wrapped_range(v, -pi, pi) (structure_model/utils.py:20-40): torch `%` is fmod, then + 2pi if the remainder is negative.
// The python-float bounds enter the fp32 kernels as their nearest fp32 values.
__device__ __forceinline__ float wrap_angle(float v) {
  constexpr float kMin = -3.14159274101257324f, kTop = 6.28318548202514648f;
  float m = fmodf(__fsub_rn(v, kMin), kTop);
  if (m != 0.f && m < 0.f) m = __fadd_rn(m, kTop);
  return __fadd_rn(m, kMin);
}
// FoldingDiff's smooth-L1 on a wrapped angle difference: h(d) = 0.5 d^2 / beta (|d| < beta), |d| - 0.5 beta otherwise; beta = pi / 10
constexpr float kAngleBeta = 0.314159265358979f;
__device__ __forceinline__ float angle_smooth_l1(float d) {
  const float ad = fabsf(d);
  return ad < kAngleBeta ? 0.5f * d * d / kAngleBeta : ad - 0.5f * kAngleBeta;
}

// ---- misc -------------------------------------------------------------------------------------------
inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
int num_sms();  // SM count of the current device (cached)

}  // namespace seqdiff
