// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM / commit).
// Everything here is device-only and header-only; used by gemm_tcgen05.cu and attn_tcgen05.cu.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

// ----------------------------------------------------------------------------------------------
// 16-bit storage type of the library.  The same sources build twice: libvl2.so stores activations / weights as bf16,
// libvl2_f16.so (-DVL2_HALF) as IEEE fp16 - the reference's own inference dtype (videollama2/__init__.py:60,
// model/__init__.py:71 load everything with torch_dtype=float16).  Every kernel moves 16-bit elements through the helpers
// below (pack_bf16 / bf16_lo / bf16_hi / unpack8 / pack8) and the CUDA conversion intrinsics, so the half build only
// re-targets those names; accumulation is fp32 either way and tcgen05.mma kind::f16 takes both input formats.
// ----------------------------------------------------------------------------------------------
#ifdef VL2_HALF
#define __nv_bfloat16 __half
#define __nv_bfloat162 __half2
#define __float2bfloat16_rn __float2half_rn
#define __bfloat162float __half2float
#define __floats2bfloat162_rn __floats2half2_rn
#define __bfloat16_as_ushort __half_as_ushort
#define VL2_UMMA_FMT 0u                          // tcgen05 instruction descriptor: A / B format F16
#define VL2_MMA_SYNC_TYPES "f16.f16"
#define VL2_MULTIMEM_TYPE "f16x2"
#define VL2_STORAGE_DTYPE 1
#else
#define VL2_UMMA_FMT 1u                          // BF16
#define VL2_MMA_SYNC_TYPES "bf16.bf16"
#define VL2_MULTIMEM_TYPE "bf16x2"
#define VL2_STORAGE_DTYPE 0
#endif

namespace vl2 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL, opt-in with VL2_PDL=1): every kernel of the library can be launched with the
// programmatic-stream-serialization attribute and starts with  pdl_launch_dependents(); ...local setup...; pdl_wait();
// so the NEXT kernel's CTAs are scheduled (and run their prologue) while this kernel's last wave drains, and a kernel
// never touches global memory before all of its predecessors have completed and flushed.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin on try_wait (HW-suspending). A bounded spin count turns a protocol bug into a trap instead of a hang,
// which matters on a GPU box we cannot attach to: a hung kernel costs the whole gpurun lease.
#ifndef VL2_MBAR_SPIN_LIMIT
#define VL2_MBAR_SPIN_LIMIT (1u << 24)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  // First poll outside the loop: ptxas puts a YIELD in front of a polling LOOP's try_wait, and a warp that yields next to
  // a sibling warp with a long run of ready instructions (the other half-row's exp2 pass, an epilogue) is not picked
  // again for ~200 cycles - even when the barrier was complete all along.  The straight-line poll carries no YIELD.
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > VL2_MBAR_SPIN_LIMIT) { asm volatile("trap;"); }
  }
}

// Wait that PARKS the thread: try_wait with a suspend-time hint, so the hardware keeps the thread asleep until the phase
// completes (or the hint expires) instead of returning to a polling loop after the short default limit.  For the roles
// that wait LONG by design (a producer for a free ring slot, the MMA issuer for the softmax warps, epilogue warps for a
// whole mainloop): their polling loops kept the SM's barrier unit so busy that every other thread's poll - even one that
// is satisfied at once - took ~200 cycles instead of ~40 (attention trace: "repeated (satisfied) S poll").
__device__ __forceinline__ bool mbar_try_wait_parked(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait_parked(bar, parity)) {
    if (++spins > VL2_MBAR_SPIN_LIMIT) { asm volatile("trap;"); }
  }
}

// Wait for two barriers at once: both polls are in flight together, so a wait that is already satisfied costs one barrier
// round trip instead of two (each poll is a few hundred cycles when eight warps hit the barrier unit at the same time).
__device__ __forceinline__ void mbar_wait2(uint64_t* bar_a, uint32_t parity_a, uint64_t* bar_b, uint32_t parity_b) {
  {   // first pair of polls outside the loop (no YIELD in front of it: see mbar_wait)
    const bool a = mbar_try_wait(bar_a, parity_a);
    const bool b = mbar_try_wait(bar_b, parity_b);
    if (a && b) return;
  }
  uint32_t spins = 0;
  for (;;) {
    const bool a = mbar_try_wait(bar_a, parity_a);
    const bool b = mbar_try_wait(bar_b, parity_b);
    if (a && b) break;
    if (++spins > VL2_MBAR_SPIN_LIMIT) { asm volatile("trap;"); }
  }
}

// wait whose acquire has CLUSTER scope: for barriers other CTAs of the cluster arrive on (release.cluster) after writing
// this CTA's shared memory through DSMEM
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0, ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (!ok && ++spins > VL2_MBAR_SPIN_LIMIT) { asm volatile("trap;"); }
  }
}

// ----------------------------------------------------------------------------------------------
// Proxy / tcgen05 fences
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// TMA store of one box from shared to global memory (bulk async-group completion).  The writers of the smem box must
// have executed fence.proxy.async (fence_proxy_async_smem) and synchronised with the issuing thread first; parts of the
// box outside the tensor are not written.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the issuing thread's bulk groups have finished READING shared memory (the source buffers may be rewritten)
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// Hint a 2-D tile of a tensor map into L2 (no smem, no barrier): issued a few k-blocks ahead of the real load so that the
// HBM latency is off the smem-stage round trip.
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* m, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(c0), "r"(c1)
               : "memory");
}
// 1-D bulk copy global -> shared (no tensor map): size and both addresses multiples of 16 bytes.
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// TMEM allocation (one full warp executes these)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ----------------------------------------------------------------------------------------------
// UMMA descriptors.
//
// Shared-memory matrix descriptor (64 bit), sm_100 flavour:
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4   [46,48) version = 1   [49,52) base offset   [61,64) layout type
// layout type: 0 none, 1 128B_base32B, 2 128B, 4 64B, 6 32B.
//
// K-major, SWIZZLE_128B (what TMA writes for a {64 x rows} bf16 box with CU_TENSOR_MAP_SWIZZLE_128B):
//   row r lives at r*128 B, its 16-byte chunks XOR-ed with (r & 7); 8-row groups are 1024 B apart => SBO = 1024.
//   LBO is ignored for swizzled K-major layouts (set to 1).  Stepping K by 16 bf16 inside the 128-B atom is
//   start_address += 32 B.
// MN-major, SWIZZLE_128B (a {64 x k-rows} box whose contiguous dim is M/N):
//   element (mn, k) lives at k*128 B + mn*2 B (swizzled by k & 7); 8-k groups 1024 B apart => SBO = 1024;
//   the next 64-wide MN atom is LBO bytes away.  Stepping K by 16 is start_address += 2048 B.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

// The same descriptor as two 32-bit words.  The start address lives in bits [0,14) of the LOW word, so stepping through a
// tile is `lo + (byte_offset >> 4)` (no carry out of the field while the address stays inside the 228 KB of shared memory)
// and the high word is a compile-time constant: an issuing thread that keeps (lo, hi) apart needs ONE uniform add per
// operand per MMA, where rebuilding the 64-bit descriptor from the address costs a dependent shift / mask / or chain of
// uniform-datapath instructions (~100 cycles per tcgen05.mma, measured in the attention kernel's timeline trace).
__host__ __device__ constexpr uint32_t umma_desc_sw128_hi(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (2u << 29);
}
__device__ __forceinline__ uint32_t umma_desc_sw128_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
// D[tmem] (+)= A[smem] * B[smem] with the descriptors given as (lo, hi) words; issued by ONE (elected) thread.
__device__ __forceinline__ void umma_bf16_ss_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                  uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// cta_group::2 form of the same (leader CTA's elected thread; operands from both CTAs' shared memory)
__device__ __forceinline__ void umma_bf16_ss_pair_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                       uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}\n"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (M = 128 rows = TMEM lanes, K along the columns, two 16-bit elements
// per 32-bit column: element k in column k / 2, even k in the low half) is read from tensor memory - no shared-memory
// traffic for it.  Issued by ONE (elected) thread.
__device__ __forceinline__ void umma_bf16_ts_lohi(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}\n"
      ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Instruction descriptor for kind::f16 with BF16 A/B and FP32 accumulate.
//   [4,6) c_format (1 = f32)  [7,10) a_format (1 = bf16)  [10,13) b_format  [15] a_major  [16] b_major
//   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (VL2_UMMA_FMT << 7) | (VL2_UMMA_FMT << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- cta_group::2 (CTA pair) variants --------------------------------------------------------------------------
// Shared addresses of a clustered launch carry the CTA rank in bit 24; clearing it addresses the same offset in the
// even ("leader") CTA of the pair (CUTLASS: Sm100MmaPeerBitMask).
static constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's mbarrier (executed by both CTAs of the pair)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar_local, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar_local) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar_local, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar_local) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar_local, int c0, int c1,
                                                 int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar_local) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// arrive on the barrier at the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar_local, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar_local)), "r"(rank)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A (128 rows from each CTA's smem) * B (N/2 rows from each CTA's smem); leader thread only
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit -> arrive on the barrier at this smem offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar_local) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar_local) & kPeerBitMask), "h"((uint16_t)3)
      : "memory");
}

// TMEM -> registers: each thread of the warp reads 32 consecutive fp32 columns of its own lane
// (lane = 32 * (warp_id % 4) + lane_id).  taddr = (lane << 16) | column.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM, same 32x32b shape (thread writes 32 consecutive columns of its lane)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
// the same store, 16 columns
__device__ __forceinline__ void tmem_st_32x32_x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// three-input maximum (one FMNMX3 on sm_100)
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// 2^x on the MUFU pipe (single instruction; inputs here are <= ~8, flush-to-zero is fine for probabilities)
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// explicit shared-space 16-byte accesses on 32-bit shared addresses (keeps the compiler from emitting generic LD/ST)
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// ----------------------------------------------------------------------------------------------
// small numeric helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
#ifdef VL2_HALF
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __half2float(__ushort_as_half((unsigned short)(u & 0xffffu))); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __half2float(__ushort_as_half((unsigned short)(u >> 16))); }
#else
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
#endif
// Two fp8 E4M3 codes (low byte = first element) -> fp32, exactly: one cvt to f16x2 (every E4M3 value, subnormals
// included, is an fp16 value) and two f16 -> f32 conversions.
__device__ __forceinline__ float2 e4m3x2_to_float2(uint32_t two_codes) {
  uint32_t h2;
  asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h2) : "h"((unsigned short)two_codes));
  float lo, hi;
  asm("cvt.f32.f16 %0, %1;" : "=f"(lo) : "h"((unsigned short)(h2 & 0xffffu)));
  asm("cvt.f32.f16 %0, %1;" : "=f"(hi) : "h"((unsigned short)(h2 >> 16)));
  return make_float2(lo, hi);
}

}  // namespace vl2
