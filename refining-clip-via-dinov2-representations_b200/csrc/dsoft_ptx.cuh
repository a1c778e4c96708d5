// Thin inline-PTX wrappers for the sm_100a features the DINO-Soft kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (TMEM alloc / mma / ld / commit) and proxy fences.
// Everything here is sm_100a-only; there is deliberately no fallback path.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace dsoft {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a fully converged warp.  The producer / MMA-issuer warps run their loops warp-uniformly and
// predicate only the issue instructions with this: inside a divergent `if (lane == 0)` the compiler cannot
// keep descriptors in uniform registers and wraps every UTCHMMA / UTMALDG in an ELECT + R2UR waterfall loop
// (measured: the issuing thread, not the tensor pipe or L2, then bounds the kernel at ~40 %).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_barrier_init() {
  // make mbarrier.init visible to the async proxy (TMA / tcgen05.commit arrive on them)
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}

// Bounded wait: a protocol bug must turn into a trap (launch failure), never into a hung GPU.
#ifndef DSOFT_SPIN_LIMIT
#define DSOFT_SPIN_LIMIT (1u << 26)
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > DSOFT_SPIN_LIMIT) {
      printf("dsoft: mbarrier timeout block=(%d,%d,%d) thread=%d bar=%u parity=%u\n", blockIdx.x,
             blockIdx.y, blockIdx.z, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ----------------------------------------------------------------------------------------------
// Proxy / tcgen05 fences
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  // generic-proxy st.shared  ->  async-proxy readers (tcgen05.mma operand fetch)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// 2-D tiled load: box lands at smem_dst, completion is signalled as tx-bytes on `bar`.
// c0 = innermost (feature) coordinate, c1 = row coordinate. Out-of-bounds elements are zero-filled.
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// Thread-block cluster
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
// shared::cta address -> shared::cluster address of the same offset in CTA `cta_rank`
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta_rank));
  return r;
}
// DSMEM bulk copy: local shared memory -> a peer CTA's shared memory, completion (tx bytes) on the
// peer's mbarrier.  Both dst and mbar are shared::cluster addresses (mapa_shared).
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes,
                                                  uint32_t mbar_cluster) {
  asm volatile(
      "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          dst_cluster),
      "r"(src_cta), "r"(bytes), "r"(mbar_cluster)
      : "memory");
}
// 1-D bulk copy global -> this CTA's shared memory (16-byte aligned, size multiple of 16), completion as tx
// bytes on a local mbarrier
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
      : "memory");
}
// all threads of all CTAs in the cluster (a plain CTA barrier when the cluster has one CTA)
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// TMEM allocation (whole warp, .sync.aligned)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_holder),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05.mma (bf16 x bf16 -> fp32 in TMEM), single CTA, both operands from shared memory
// ----------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor for a SWIZZLE_128B tile whose rows are 128 bytes (64 bf16):
//   bits [0,14)  start address >> 4
//   bits [16,30) leading-dimension byte offset >> 4
//   bits [32,46) stride-dimension byte offset >> 4
//   bits [46,48) descriptor version (1 on sm_100)
//   bits [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// Instruction descriptor for kind::f16 with bf16 operands and fp32 accumulation.
//   bits [4,6) c_format (1 = f32), [7,10) a_format (1 = bf16), [10,13) b_format (1 = bf16),
//   bit 15 a_major (0 = K-major), bit 16 b_major (1 = MN-major), [17,23) N>>3, [24,29) M>>4
//   f16 = 1 selects fp16 (format 0) for BOTH operands: the hardware rejects mixed fp16 x bf16
//   (measured: cudaErrorIllegalInstruction), so A and B always share one format.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major,
                                                       int f16 = 0) {
  return (1u << 4) | ((f16 ? 0u : 1u) << 7) | ((f16 ? 0u : 1u) << 10) |
         (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Arrives on `bar` once every tcgen05.mma issued so far by this thread has completed.
// (Implies tcgen05.fence::before_thread_sync.)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}

// Multicast commit: arrives on the mbarrier at this offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          bar),
      "h"(cta_mask)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// cta_group::2 variants: a pair of CTAs (cluster ranks 2k, 2k+1) drives one M=256 MMA.  Each CTA holds its
// own 128 rows of A and half of the N rows of B at the SAME shared-memory offsets; the leader (even rank)
// issues; accumulator rows 0..127 land in the leader's TMEM, 128..255 in the peer's, same TMEM address.
// Every tcgen05 instruction of a kernel must use one cta_group, hence the compile-time parameter.
// ----------------------------------------------------------------------------------------------
template <int CG>
__device__ __forceinline__ void tmem_alloc_cg(uint32_t smem_holder, uint32_t ncols) {
  if constexpr (CG == 1) {
    tmem_alloc(smem_holder, ncols);
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_holder),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc_cg(uint32_t taddr, uint32_t ncols) {
  if constexpr (CG == 1) {
    tmem_dealloc(taddr, ncols);
  } else {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  }
}
template <int CG>
__device__ __forceinline__ void umma_cg(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  if constexpr (CG == 1) {
    umma_bf16(tmem_d, adesc, bdesc, idesc, accumulate);
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}"
        :
        : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// commit: CG == 2 arrives on the barrier at this offset in BOTH CTAs of the pair (`pair_mask` = 0b11 << 2k)
template <int CG>
__device__ __forceinline__ void umma_commit_cg(uint32_t bar, uint16_t pair_mask = 3) {
  if constexpr (CG == 1) {
    umma_commit(bar);
  } else {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            bar),
        "h"(pair_mask)
        : "memory");
  }
}
// TMA load issued by either CTA of a pair; completion bytes are credited to `bar_cluster`, a shared::cluster
// address (mapa_shared) of the mbarrier in the pair's leader.
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar_cluster,
                                                int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
// Arrive on an mbarrier of another CTA of the cluster (address from mapa_shared) without release semantics: a
// .release arrive waits until every earlier global store of the thread has been performed at cluster scope (MEMBAR),
// which stalls an epilogue that streams tiles to HBM.  Valid when the barrier only hands back TMEM (reads completed
// by tcgen05.wait::ld + fence::before_thread_sync), not memory.
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}

// Read-only 16-byte global load that the compiler may not sink towards its first use (software prefetch of
// per-column statistics ahead of the tile they belong to).
__device__ __forceinline__ float4 ldg_nc_v4_volatile(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (one row per thread).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Same for 16 and 8 consecutive columns (epilogues whose other live registers leave no room for 32).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// Split form for software pipelining: issue the load of the NEXT 32-column chunk, compute on the current one, and
// only then wait.  tcgen05.wait::ld covers every earlier tcgen05.ld of the thread; the registers are passed through
// the wait as in/out operands so that the compiler cannot move a consumer above it.
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                 "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                 "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// 16 lanes x 256 bits, four repeats = a 16-row x 32-column fp32 block per instruction.  Thread t holds, for the
// 8-column group j = 0..3:  r[4j], r[4j+1] = row (t / 4), columns 8j + 2 (t % 4) + {0, 1};  r[4j+2], r[4j+3] = row
// (t / 4) + 8, same columns (the accumulator-fragment layout of mma.m16n8).  The lane field of `taddr` selects the
// first of the 16 lanes (a warp reaches the 32 lanes of its quadrant: + 16 for the second half).
__device__ __forceinline__ void tmem_ld16x256_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15])
               :
               : "memory");
}

// L2 eviction policies for bulk-tensor traffic.  The logit-gradient kernels write gigabytes of G tiles that are not
// read again before the gradient GEMM, next to a few hundred megabytes of operands that every CTA re-reads: without
// hints the stores pushed the operands out of L2 (hit rate 38 - 57 %, MMA issuer starved for operands).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_2d_2sm_hint(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar_cluster,
                                                     int32_t c0, int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* map, uint32_t smem_src, int c0, int c1,
                                                  uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;"
               :: "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_src), "r"(c0), "r"(c1), "l"(policy)
               : "memory");
}

__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all but the N most recent bulk groups of this thread have finished READING their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// x = m * 2^e (normal, positive): mant12(x) = m in [1, 2), pow2_of(x) = 2^e; both exact bit operations.
// Zero maps to (1, 0), +inf to (1, inf): callers only meet those on padded / masked entries.
__device__ __forceinline__ float mant12(float x) {
  return __uint_as_float((__float_as_uint(x) & 0x007fffffu) | 0x3f800000u);
}
__device__ __forceinline__ float pow2_of(float x) { return __uint_as_float(__float_as_uint(x) & 0x7f800000u); }

// Register reallocation between warpgroups (the epilogue warps of the soft kernels hold a 128-column strip of
// teacher weights per thread; the TMA / MMA / allocator warps need almost nothing).
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// Named barrier over a subset of the block's warps (nthreads a multiple of 32; id 0 is __syncthreads).
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Warp-wide float maximum / minimum in one instruction (sm_100a: redux.sync on f32, result in a uniform register)
__device__ __forceinline__ float warp_max_f32(float x) {
  float r;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float warp_min_f32(float x) {
  float r;
  asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(x));
  return r;
}

// two fp32 -> packed bf16x2 (lo = first argument), round-to-nearest-even
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// two fp32 -> packed f16x2 (lo = first argument)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}

}  // namespace dsoft
