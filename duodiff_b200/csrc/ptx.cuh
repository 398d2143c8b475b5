// sm_100a PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM), misc.
// Hand-written inline PTX; no CUTLASS dependency.  Bit layouts of the UMMA shared-memory
// descriptor and instruction descriptor follow the PTX ISA "tcgen05" chapter.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ddb {

// Device-side step state -- the live sample / row counts of the early-exit compaction, slot maps, exit indices, the
// step counter -- is rewritten by one kernel of a step and read by the next.  With programmatic dependent launch the
// reader's CTAs are resident BEFORE the writer has finished: if anything on the same SM reads the line in that window
// (the writer itself, e.g. ee_decide_kernel reading ee_n[0] before its last CTA rewrites ee_n[2]), the reader's load
// after griddepcontrol.wait hits the stale L1 line (seen on B200: ee_move_kernel read n_exit = 0 and skipped the move).
// All such state is therefore read through L2.
__device__ __forceinline__ int ld_state(const int* p) { return __ldcg(p); }
__device__ __forceinline__ unsigned long long ld_state(const unsigned long long* p) { return __ldcg(p); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// non-blocking probe (the single MMA-issuing thread polls several barriers)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// try_wait with an explicit suspend-time hint (ns): the warp sleeps in hardware until the phase completes or the time
// limit passes, instead of returning to a software spin loop that competes for its scheduler's issue slots
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
        : "memory");
    return ok != 0;
}
// Bounded spin: a protocol bug traps (launch failure) instead of hanging the GPU.
#ifndef DDB_SPIN_LIMIT
#define DDB_SPIN_LIMIT (1u << 26)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > DDB_SPIN_LIMIT) __trap();
    }
}
// long waits (hundreds of clocks or more): sleep in hardware, 20 us per try
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait_hint(bar, parity, 20000u)) {
        if (++spins > (1u << 20)) __trap();
    }
}

// ----------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
// 2-D tile load global -> shared, completion signalled on an mbarrier (complete_tx bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
        "[%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// 4-D tile load (NHWC activations of the autoencoder's implicit-GEMM convolutions: coordinates {c, x, y, b}; signed
// coordinates outside the tensor are zero-filled, which is the convolution's zero padding).
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
        "%6}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// 5-D tile load (the stride-2 view {(q, c), x/2, p, y/2, b} of NHWC activations: the encoder's Downsample conv).
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
        "%6, %7}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* tm, const void* smem_src, int c0, int c1, int c2,
                                             int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tm)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}
// 2-D tile store shared -> global (bulk async group).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tm)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tm)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
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
// generic-proxy writes to smem -> visible to the async proxy (TMA store / UMMA operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// L2 eviction-priority policies for TMA traffic (createpolicy): evict_first for operands that are dead after this read,
// evict_last for tensors the next kernel re-reads.
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
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* tm, const void* smem_src, int c0, int c1,
                                                  uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(
                     reinterpret_cast<uint64_t>(tm)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(policy)
                 : "memory");
}

// ----------------------------------------------------------------------------- programmatic dependent launch
// Every kernel of the sampling step is launched with programmaticStreamSerialization: it may become resident while its
// predecessor is still draining.  pdl_launch_dependents() lets the successor's CTAs be scheduled as soon as this
// grid's CTAs free their SMs; pdl_wait() blocks until the predecessor grid has completed and its writes are visible.
// It must precede the first access to anything a previous kernel wrote (and any write a previous kernel may still
// read).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ----------------------------------------------------------------------------- named barriers
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ----------------------------------------------------------------------------- tcgen05 / TMEM
template <uint32_t NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
                 "n"(NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16/fp16 inputs with fp32 accumulate.
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand from TMEM (bf16 packed 2/column), B from smem.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once every tcgen05 op previously issued by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive columns: thread i of the warp receives row (lane base + i), columns [c, c+32).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// UMMA shared-memory matrix descriptor (64-bit):
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset>>4 [46,48) version (1 on sm_100)
//   [49,52) base offset               [61,64) swizzle: 0 none, 2 = 128B, 4 = 64B, 6 = 32B
// K-major operand, 128-byte swizzle, tile rows of exactly 128 B (64 bf16): 8-row atoms 1024 B apart.
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);  // start address
    d |= static_cast<uint64_t>(0) << 16;                     // LBO unused: one swizzle atom along K
    d |= static_cast<uint64_t>(1024 >> 4) << 32;             // SBO: 8 rows * 128 B
    d |= static_cast<uint64_t>(1) << 46;                     // descriptor version
    d |= static_cast<uint64_t>(2) << 61;                     // SWIZZLE_128B
    return d;
}
// MN-major operand (e.g. V[keys, head_dim] used as B = V^T), 128-byte swizzle, 64 bf16 along MN per row:
// K index = smem row (128 B apart), 8-row atoms 1024 B apart (SBO); one atom along MN (LBO unused).
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>(1024 >> 4) << 16;  // LBO (unused when MN extent is one atom)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;  // SBO: next group of 8 K rows
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32.
//   [4,6) D fmt (1 = f32)  [7,10) A fmt (1 = bf16)  [10,13) B fmt  [15] A major  [16] B major (0 = K)
//   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major = 0,
                                                        uint32_t b_mn_major = 0) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((N >> 3) << 17) |
           ((M >> 4) << 24);
}

// ----------------------------------------------------------------------------- clusters / cta_group::2
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem offset in the even (leader) CTA of a CTA pair
__device__ __forceinline__ uint32_t leader_smem_addr(const void* p) { return smem_u32(p) & 0xFEFFFFFFu; }
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
template <uint32_t NCOLS>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_holder) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
                 "n"(NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t NCOLS>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// CTA-pair MMA (M = 256 across the two CTAs), issued by one thread of the leader CTA.
__device__ __forceinline__ void umma_f16_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the barrier at this smem offset in every CTA of `mask` once the pair's prior MMAs have completed
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
                     "r"(smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
// TMA load into this CTA's smem whose completion bytes are credited to the leader CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_2cta_hint(void* smem_dst, const CUtensorMap* tm, uint32_t leader_bar, int c0,
                                                      int c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_2cta(void* smem_dst, const CUtensorMap* tm, uint32_t leader_bar, int c0,
                                                 int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
        "[%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}

// ----------------------------------------------------------------------------- packed fp32x2 math (FFMA2 on sm_100)
typedef uint64_t f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f32x2 f2_pack_u(uint32_t lo, uint32_t hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 f2_splat(float v) { return f2_pack(v, v); }
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint32_t f2_to_bf16x2(f32x2 v) {
    float lo, hi;
    f2_unpack(v, lo, hi);
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// ----------------------------------------------------------------------------- misc
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// GELU (exact-erf form, nn.GELU default) as 0.5 x (1 + tanh(x q(x^2))) with q fitted to the erf form on [-8, 8]
// (max abs deviation 2.5e-5 before the tanh.approx error of ~2^-11 relative; well inside bf16 output rounding).
// x^2 is clamped so the cubic-in-x^2 inner polynomial stays monotone for any input.
__device__ __forceinline__ f32x2 gelu_fast2(f32x2 x) {
    float a, b;
    f2_unpack(f2_mul(x, x), a, b);
    const f32x2 x2 = f2_pack(fminf(a, 64.f), fminf(b, 64.f));
    const f32x2 q = f2_fma(f2_fma(f2_splat(-0.00035151747709065645f), x2, f2_splat(0.0370056505644417f)), x2,
                           f2_splat(0.7975078789081762f));
    const f32x2 hx = f2_mul(x, f2_splat(0.5f));
    f2_unpack(f2_mul(x, q), a, b);
    return f2_fma(hx, f2_pack(tanh_approx(a), tanh_approx(b)), hx);
}
__device__ __forceinline__ float gelu_fast(float x) {
    const float x2 = fminf(x * x, 64.f);
    const float q = fmaf(fmaf(-0.00035151747709065645f, x2, 0.0370056505644417f), x2, 0.7975078789081762f);
    const float hx = 0.5f * x;
    return fmaf(hx, tanh_approx(x * q), hx);
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

}  // namespace ddb
