// Thin inline-PTX wrappers for the sm_100a features the HGEMM kernel uses:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld), cluster.
// Nothing here depends on CUTLASS/CuTe; encodings were cross-checked against the PTX ISA
// and the SASS that nvcc 12.9 emits (UTCHMMA / UTMALDG / UTMASTG / LDTM / UTCBAR).
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#ifndef B200_HGEMM_WATCHDOG
#define B200_HGEMM_WATCHDOG 1   // bounded mbarrier spins: a protocol bug traps instead of hanging the GPU
#endif

namespace b200 {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- cluster
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\t"
               "barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_addr` in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on a barrier that lives in (possibly) another CTA of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#if B200_HGEMM_WATCHDOG
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {   // seconds of spinning: a phase/count bug, not a slow tile
      printf("b200_hgemm watchdog: block %d thread %d stuck on mbarrier 0x%x parity %u\n",
             (int)blockIdx.x, (int)threadIdx.x, bar, parity);
      __trap();
    }
  }
#else
  while (!mbar_try_wait(bar, parity)) {}
#endif
}

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tile load global -> this CTA's smem, completion bytes on `bar`.
// kCtaGroup == 2: `bar` may be a shared::cluster address inside the pair (the leader's barrier).
template <int kCtaGroup>
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* tmap, uint32_t bar,
                                            int32_t c0, int32_t c1) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
  }
}
// multicast variant: the same box lands at the same smem offset of every CTA in `mask`,
// each destination CTA's barrier (same offset) receives the bytes.
template <int kCtaGroup>
__device__ __forceinline__ void tma_load_2d_mcast(uint32_t smem_dst, const void* tmap, uint32_t bar,
                                                  int32_t c0, int32_t c1, uint16_t mask) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
        : "memory");
  }
}
// L2 eviction-priority policies for TMA loads (createpolicy encodings, as used by CUTLASS' TMA::CacheHintSm90)
constexpr uint64_t kL2EvictNormal = 0x1000000000000000ull;
constexpr uint64_t kL2EvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kL2EvictLast = 0x14F0000000000000ull;

template <int kCtaGroup>
__device__ __forceinline__ void tma_load_2d_hint(uint32_t smem_dst, const void* tmap, uint32_t bar,
                                                 int32_t c0, int32_t c1, uint64_t hint) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
  }
}
template <int kCtaGroup>
__device__ __forceinline__ void tma_load_2d_mcast_hint(uint32_t smem_dst, const void* tmap, uint32_t bar,
                                                       int32_t c0, int32_t c1, uint16_t mask, uint64_t hint) {
  if constexpr (kCtaGroup == 1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5, %6;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "h"(mask), "l"(hint)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5, %6;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "h"(mask), "l"(hint)
        : "memory");
  }
}

// 1-D bulk copy global -> this CTA's smem (bytes % 16 == 0, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_load_1d(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(bar)
               : "memory");
}
// order earlier generic-proxy accesses (made visible to this thread) before later async-proxy accesses
__device__ __forceinline__ void fence_proxy_async_all() {
  asm volatile("fence.proxy.async;" ::: "memory");
}
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int kPending>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------- tcgen05: TMEM management
template <int kCtaGroup>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_result_addr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_result_addr), "r"(ncols) : "memory");
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---------------------------------------------------------------- tcgen05: MMA + commit
// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread for the CTA (pair).
template <int kCtaGroup>
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, uint32_t accumulate) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrive once all previously issued MMAs of this thread have completed.
// (implies tcgen05.fence::before_thread_sync)
template <int kCtaGroup>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 ::"r"(bar) : "memory");
  else
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 ::"r"(bar) : "memory");
}
// same, but the arrive is delivered to the barrier at this offset in every CTA of `mask`
template <int kCtaGroup>
__device__ __forceinline__ void umma_commit_mcast(uint32_t bar, uint16_t mask) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"(mask) : "memory");
  else
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"(mask) : "memory");
}

// ---------------------------------------------------------------- tcgen05: TMEM -> registers
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives lane (base+i).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// fp16 accumulators: 64 consecutive columns (16 significant bits each) packed 2-per-register
__device__ __forceinline__ void tmem_ld_32x32b_x32_pack16(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// fp16 accumulators, 32 consecutive columns packed into 16 registers
__device__ __forceinline__ void tmem_ld_32x32b_x16_pack16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.pack::16b.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
__device__ __forceinline__ void grid_dependency_wait() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
__device__ __forceinline__ void grid_dependency_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ---------------------------------------------------------------- misc
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
// load from the shared memory of any CTA in the cluster (address from mapa)
__device__ __forceinline__ float4 ld_dsmem_v4f(uint32_t cluster_addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(cluster_addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_v4f(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float4 ld_shared_v4f(uint32_t addr) {
  float4 v;
  // reads data published by an mbarrier wait (async-proxy bulk copies): must not be hoisted above it
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t pack_f16x2_rn(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);   // cvt.rn.f16x2.f32: one rounding per element
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);   // cvt.rn.bf16x2.f32
  return *reinterpret_cast<uint32_t*>(&h);
}
// the output element type follows the operands': fp16 in -> fp16 out, bf16 in -> bf16 out
template <bool kBf16>
__device__ __forceinline__ uint32_t pack_out_x2_rn(float lo, float hi) {
  if constexpr (kBf16) return pack_bf16x2_rn(lo, hi);
  else return pack_f16x2_rn(lo, hi);
}


// ---------------------------------------------------------------- global memory, L2-only (data exchanged between CTAs)
__device__ __forceinline__ void st_global_cg_v4(uint4* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.cg.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_global_cg_v4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.cg.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

}  // namespace ptx
}  // namespace b200
