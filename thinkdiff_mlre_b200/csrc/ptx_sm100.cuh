// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (TMEM alloc,
// MMA, commit, ld) and the shared-memory / instruction descriptors the tensor core consumes.
// Nothing here is ThinkDiff-specific; the aligner kernels in gemm_sm100.cuh are built from these.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace td {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Arrive on the barrier at the same smem offset in CTA `cta` of this cluster.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n .reg .b32 ra;\n"
      " mapa.shared::cluster.u32 ra, %0, %1;\n"
      " mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n}" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      " selp.b32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n"
      " mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
      " selp.b32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Store a 32-bit value into the same shared-memory location of CTA `cta` of this cluster (DSMEM).
__device__ __forceinline__ void st_shared_cluster_s32(int* local_addr, uint32_t cta, int value) {
  asm volatile(
      "{\n .reg .b32 ra;\n"
      " mapa.shared::cluster.u32 ra, %0, %1;\n"
      " st.shared::cluster.s32 [ra], %2;\n}" ::"r"(smem_u32(local_addr)),
      "r"(cta), "r"(value)
      : "memory");
}
// A pipeline wait that cannot hang the GPU: if a barrier does not flip within ~4 s the kernel
// traps, which surfaces as a launch failure on the host instead of a wedged device.
#ifndef TD_MBAR_TIMEOUT_NS
#define TD_MBAR_TIMEOUT_NS 4000000000ull
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = global_timer_ns();
  while (!mbar_try_wait(bar, parity)) {
    if (global_timer_ns() - t0 > TD_MBAR_TIMEOUT_NS) {
      printf("td: mbarrier timeout block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}

// Same, with cluster-scope acquire: the barrier may have been arrived on by (and orders data written by) the peer CTA.
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const uint64_t t0 = global_timer_ns();
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (global_timer_ns() - t0 > TD_MBAR_TIMEOUT_NS) {
      printf("td: cluster mbarrier timeout block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- global-memory flags (stream-K fix-up, peer exchange)
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Wait until another CTA of this grid has stored a non-zero value (release) to *p: relaxed polls, one acquire fence at the end
// (an acquire load per iteration would invalidate L1 every time). Same 4 s trap as the mbarrier waits.
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void spin_until_set(const int* p) {
  if (ld_relaxed_gpu(p) == 0) {
    const uint64_t t0 = global_timer_ns();
    while (ld_relaxed_gpu(p) == 0) {
      __nanosleep(64);
      if (global_timer_ns() - t0 > TD_MBAR_TIMEOUT_NS) {
        printf("td: stream-K flag timeout block %d thread %d\n", blockIdx.x, threadIdx.x);
        __trap();
      }
    }
  }
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start while the previous kernel of its stream
// is still running. grid_dependency_wait() blocks until that kernel has completed and its memory is visible; without the
// attribute it returns at once. It only orders a kernel after its immediate predecessor, so every kernel launched with the
// attribute must call it on every path -- otherwise it could finish before its predecessor, and its own successor's wait would
// no longer cover that predecessor.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Let the next kernel of the stream start launching (its CTAs run up to their grid_dependency_wait()).
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- cluster
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- TMA
// A tensor map that lives in GLOBAL memory (not a __grid_constant__ parameter) must be acquired through the tensormap proxy by
// the thread that is going to issue TMA operations with it.
__device__ __forceinline__ void fence_tensormap_acquire(const CUtensorMap* m) {
  asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" ::"l"(m) : "memory");
}

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// cta_group::2 form: both CTAs of a pair issue it, the bytes are signalled on the LEADER CTA's barrier
// (bit 24 of a shared::cluster address selects the peer; clearing it addresses CTA rank 0 of the pair).
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
// Same box, added element-wise into global memory (fp32 tensor map): out += box.
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <int CTAS>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  if constexpr (CTAS == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
}
template <int CTAS>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (CTAS == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int CTAS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (CTAS == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; bf16 inputs, fp32 accumulate. Issued by ONE thread.
template <int CTAS>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  if constexpr (CTAS == 1)
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
        " tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
        " tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Make `bar` flip once every tcgen05.mma issued so far by this thread has finished reading smem and
// writing TMEM. (Implies tcgen05.fence::before_thread_sync.) For a pair, `mask` names the CTAs whose
// barrier (same smem offset) receives the arrive.
template <int CTAS>
__device__ __forceinline__ void umma_commit(uint64_t* bar, uint16_t mask = 3) {
  if constexpr (CTAS == 1)
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  else
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"(mask)
        : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns; thread i receives lane
// (32*(warp%4) + i), v[j] = column (col0 + j).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- descriptors
// Instruction descriptor for kind::f16 with bf16 A/B and fp32 accumulate
// (bit layout: c_format[4,6) a_format[7,10) b_format[10,13) a_major[15] b_major[16] N>>3 [17,23) M>>4 [24,29)).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int umma_m, int umma_n, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(a_mn_major) << 15) | (uint32_t(b_mn_major) << 16) |
         (uint32_t(umma_n >> 3) << 17) | (uint32_t(umma_m >> 4) << 24);
}
// Shared-memory matrix descriptor, 128-byte swizzle, sm_100 version bit set.
//   start address, leading byte offset (LBO) and stride byte offset (SBO) are stored >> 4.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(lbo_bytes >> 4) << 16) | (uint64_t(sbo_bytes >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}

// ---------------------------------------------------------------- small math / packing helpers
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// Round two fp32 values to bf16 (round-to-nearest-even) with ONE packed conversion on the ALU pipe and get them back as fp32:
// the scalar form (F2F.BF16.F32) is an XU-pipe instruction -- quarter rate, the pipe the GELU's MUFU ops need.
__device__ __forceinline__ uint32_t bf16_round2(float& a, float& b) {
  const uint32_t p = pack_bf16x2(a, b);
  a = bf16lo(p);
  b = bf16hi(p);
  return p;
}
// MUFU ops without the denormal-range scaling the libm-style wrappers add (3-4 extra instructions each): the arguments here
// are never in those ranges (ex2: x <= 0, flushing a denormal result to zero is exact enough; rcp: the argument is >= 1).
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Fast GELU(erf) for the GEMM epilogues. Phi(-|x|) = 0.5 erfc(|x| / sqrt 2) by Abramowitz-Stegun 7.1.26
// (|abs error| <= 7.5e-8 on Phi), sharing ONE exponential e^{-x^2/2} between the cdf and the pdf:
// 2 MUFU (ex2, rcp) + 12 FMA-pipe ops per element instead of erff's ~45. Outputs are rounded to bf16 afterwards.
__device__ __forceinline__ float normal_cdf_pdf(float x, float& pdf) {
  const float e = ex2_approx((-0.72134752044448170368f * x) * x);            // e^{-x^2/2}
  const float t = rcp_approx(fmaf(0.3275911f * 0.70710678118654752440f, fabsf(x), 1.0f));
  float poly = fmaf(t, 0.5f * 1.061405429f, 0.5f * -1.453152027f);           // (the 0.5 of Phi is folded into the coefficients)
  poly = fmaf(t, poly, 0.5f * 1.421413741f);
  poly = fmaf(t, poly, 0.5f * -0.284496736f);
  poly = fmaf(t, poly, 0.5f * 0.254829592f);
  const float q = (t * poly) * e;                                            // Phi(-|x|)
  pdf = 0.39894228040143267794f * e;
  return x >= 0.f ? 1.0f - q : q;
}
__device__ __forceinline__ float gelu_fast(float x) {
  float pdf;
  return x * normal_cdf_pdf(x, pdf);
}
__device__ __forceinline__ float gelu_grad_fast(float x) {
  float pdf;
  const float cdf = normal_cdf_pdf(x, pdf);
  return fmaf(x, pdf, cdf);
}

// gelu_new (transformers NewGELUActivation, T5's gated-gelu FFN): 0.5 x (1 + tanh u), u = sqrt(2/pi) (x + 0.044715 x^3). With
// s = 0.5 (1 + tanh u) = 1 / (1 + e^{-2u}) this is x * s, and d/dx = s + x * 2 s (1 - s) u'. Both come from ONE exponential
// e = e^{-2|u|} <= 1 and r = 1 / (1 + e): s = r for u >= 0, e r for u < 0, and s (1 - s) = e r^2 either way -- no cancellation and
// no overflow at any x, |error| about 1e-7. (tanh.approx.f32 is only good to about 2^-11, close enough to half a bf16 ulp to flip
// the rounding of the outputs.)
__device__ __forceinline__ void gelu_tanh_gate(float x, float& s, float& ds) {
  const float x2 = x * x;
  const float u = 0.79788456080286535588f * fmaf(0.044715f * x2, x, x);
  const float e = ex2_approx(-2.88539008177792681472f * fabsf(u));  // e^{-2|u|}
  const float r = rcp_approx(1.0f + e);
  s = u >= 0.f ? r : e * r;
  ds = 2.0f * (e * r * r) * (0.79788456080286535588f * fmaf(3.0f * 0.044715f, x2, 1.0f));
}
__device__ __forceinline__ float gelu_tanh(float x) {
  float s, ds;
  gelu_tanh_gate(x, s, ds);
  return x * s;
}
// Derivative of gelu_tanh at x; the value gelu_tanh(x) goes to `gelu` (the backward needs both).
__device__ __forceinline__ float gelu_tanh_grad(float x, float& gelu) {
  float s, ds;
  gelu_tanh_gate(x, s, ds);
  gelu = x * s;
  return fmaf(x, ds, s);
}

// nn.GELU(approximate='none'): 0.5 x (1 + erf(x / sqrt 2)), and its derivative (libm-accurate forms).
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

}  // namespace td
