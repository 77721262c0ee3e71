// fm_ptx.cuh -- thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM),
// scoped acquire/release accesses used by the cross-CTA and cross-GPU flag protocol.
// Hand-written for this project (no CUTLASS/CuTe on the hot path -- BASELINE.json north_star).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fm {

// ----------------------------------------------------------------------------------------------------------------
// bounded spinning: every wait in the kernel gives up after `timeout_ns`, records why in a host-mapped debug record
// and traps, so a protocol bug or a dead peer ends the launch with an error instead of hanging the GPU.
// ----------------------------------------------------------------------------------------------------------------
struct DebugRecord {          // lives in pinned, device-mapped host memory (readable after a trap)
    unsigned int code;        // FM_TRAP_* below (0 = none)
    unsigned int block;
    unsigned int thread;
    unsigned int info0;
    unsigned int info1;
    unsigned int info2;
    unsigned long long waited_ns;
};

enum : unsigned int {
    FM_TRAP_NONE = 0,
    FM_TRAP_MBAR_FULL = 1,
    FM_TRAP_MBAR_EMPTY = 2,
    FM_TRAP_MBAR_TMEM_FULL = 3,
    FM_TRAP_MBAR_TMEM_EMPTY = 4,
    FM_TRAP_MBAR_SCHED_FULL = 5,
    FM_TRAP_MBAR_SCHED_EMPTY = 6,
    FM_TRAP_GRID_BARRIER = 7,
    FM_TRAP_RECV_FLAG = 8,
    FM_TRAP_G0_DONE = 9,
    FM_TRAP_RET_FLAG = 10,
    FM_TRAP_RECV_ROWS = 11,
    FM_TRAP_MBAR_PUB = 12,
};

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __noinline__ void fm_trap(DebugRecord* dbg, unsigned int code, unsigned int i0, unsigned int i1,
                                     unsigned int i2, unsigned long long waited) {
    if (dbg != nullptr) {  // plain stores to pinned host memory (no PCIe atomics needed); first writer wins loosely
        volatile DebugRecord* d = dbg;
        if (d->code == 0u) {
            d->block = blockIdx.x;
            d->thread = threadIdx.x;
            d->info0 = i0;
            d->info1 = i1;
            d->info2 = i2;
            d->waited_ns = waited;
            d->code = code;
            __threadfence_system();
        }
    }
    __trap();
}

struct SpinGuard {  // cheap: reads %globaltimer only every 256 polls
    unsigned long long t0 = 0;
    unsigned int polls = 0;
    __device__ __forceinline__ void tick(DebugRecord* dbg, unsigned long long timeout_ns, unsigned int code,
                                         unsigned int i0, unsigned int i1, unsigned int i2) {
        if ((++polls & 255u) == 0u) {
            const unsigned long long now = globaltimer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > timeout_ns) fm_trap(dbg, code, i0, i1, i2, now - t0);
        }
    }
};

// ----------------------------------------------------------------------------------------------------------------
// shared-memory addressing + mbarrier
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
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
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, DebugRecord* dbg,
                                          unsigned long long timeout_ns, unsigned int code, unsigned int info) {
    SpinGuard g;
    while (!mbar_try_wait(bar, parity)) g.tick(dbg, timeout_ns, code, info, parity, 0);
}

// ----------------------------------------------------------------------------------------------------------------
// proxy / memory fences
// ----------------------------------------------------------------------------------------------------------------
// generic-proxy global writes <-> async-proxy (TMA) global reads
__device__ __forceinline__ void fence_proxy_async_global() {
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------------------------
// scoped loads/stores/reductions for flags and counters
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_sys_add_u32(unsigned int* p, unsigned int v) {  // also on peer-mapped addresses
    asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_gpu_add_u32(unsigned int* p, unsigned int v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int atom_acq_rel_gpu_add_u32(unsigned int* p, unsigned int v) {
    unsigned int old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ unsigned long long atom_acq_rel_gpu_add_u64(unsigned long long* p,
                                                                       unsigned long long v) {
    unsigned long long old;
    asm volatile("atom.acq_rel.gpu.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
    return old;
}

// 16-byte global accesses (coalesced row copies, also valid on NVLink peer-mapped addresses)
__device__ __forceinline__ uint4 ld_global_nc_v4(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_global_v4(const void* p) {  // coherent path (data written during this launch)
    uint4 v;
    asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p)
                 : "memory");
    return v;
}
__device__ __forceinline__ int4 ld_global_cg_i4(const void* p) {   // L2-coherent (data written by other SMs in this launch)
    int4 v;
    asm volatile("ld.global.cg.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_global_v4(void* p, const uint4& v) {
    asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}

// 8 x bf16 element-wise add into global memory (REDG.E.ADD.BF16x8.RN): round-to-nearest-even like a bf16 atomicAdd,
// no return value; valid on peer-mapped addresses (NVLink atomics)
__device__ __forceinline__ void red_add_bf16x8(void* p, const uint4& v) {
    asm volatile("red.relaxed.sys.global.add.noftz.v4.bf16x2 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y),
                 "r"(v.z), "r"(v.w)
                 : "memory");
}

// ----------------------------------------------------------------------------------------------------------------
// TMA: 2-D tiled bulk tensor load, global -> shared, completion on an mbarrier (complete_tx::bytes)
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// 1-D bulk copies through the TMA engine (no tensor map): contiguous global -> shared with mbarrier completion, and
// shared -> global (also peer-mapped) tracked with bulk async-groups
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// shared-memory only: generic-proxy accesses to smem <-> async-proxy (TMA) accesses to the same smem; does not wait for
// the thread's outstanding global stores
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// L2 prefetch of a tensor tile (no smem destination, no barrier): hides HBM latency for k-blocks the pipeline will
// request a few steps later
__device__ __forceinline__ void tma_prefetch_l2_2d(const void* tmap, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(tmap), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int32_t c0, int32_t c1,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// ----------------------------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA issue, commit, TMEM loads
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {  // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16 inputs with fp32 accumulation
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives row (lane base + i), columns [c, c+32)
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


// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

// ----------------------------------------------------------------------------------------------------------------
// thread-block clusters / CTA pairs (cta_group::2): the two CTAs of a cluster run one 256-row UMMA together
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of every CTA in the cluster
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `cta` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {  // arrive on CTA `cta`'s copy
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(mapa_shared(smem_u32(bar), cta))
                 : "memory");
}
// barrier-only signal to another CTA (no data published by this thread): default semantics, no cluster-scope release
// fence (a .release.cluster arrive per k-block made the CTA-pair pipeline ~2x slower)
__device__ __forceinline__ void mbar_arrive_cluster_plain(uint64_t* bar, uint32_t cta) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(mapa_shared(smem_u32(bar), cta)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {  // acquire at cluster scope
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, DebugRecord* dbg,
                                                  unsigned long long timeout_ns, unsigned int code, unsigned int info) {
    SpinGuard g;
    while (!mbar_try_wait_cluster(bar, parity)) g.tick(dbg, timeout_ns, code, info, parity, 1);
}
__device__ __forceinline__ void st_shared_cluster_v4(uint32_t cluster_addr, const uint4& v) {
    asm volatile("st.shared::cluster.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(cluster_addr), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}
// TMA load issued by either CTA of a pair; completion bytes are credited to the mbarrier at `bar_cluster_addr`, a
// shared::cluster address (mapa_shared(smem_u32(bar), 0) = the LEADER CTA's copy of the barrier)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, int32_t c0, int32_t c1,
                                                 uint32_t bar_cluster_addr) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {  // same warp id in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 256 x N x 16 MMA across the CTA pair (issued by the leader only): rows 0-127 accumulate in the leader's TMEM, rows
// 128-255 in the peer's; A comes from each CTA's own smem, B rows [0,N/2) from the leader's smem and [N/2,N) from the peer's
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {  // arrives on the barrier at this offset in BOTH CTAs
    const unsigned short mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}

// ----------------------------------------------------------------------------------------------------------------
// UMMA descriptors (PTX ISA "tcgen05 matrix / instruction descriptors")
// ----------------------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor for a K-major bf16 operand tile stored as rows of 128 bytes (64 bf16) with the
// 128-byte swizzle TMA writes (CU_TENSOR_MAP_SWIZZLE_128B):
//   bits  0-13  start address >> 4            bits 16-29  leading-dim byte offset >> 4 (unused for swizzled K-major)
//   bits 32-45  stride-dim byte offset >> 4 = 1024 B (8 rows x 128 B swizzle atom) >> 4
//   bits 46-47  descriptor version = 1 (sm_100)     bits 61-63  layout: 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1024u >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor, kind::f16: D fp32 (bits 4-5 = 1), A/B bf16 (bits 7-9 / 10-12 = 1), both K-major
// (bits 15/16 = 0), N >> 3 at bits 17-22, M >> 4 at bits 24-28.
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(uint32_t M, uint32_t N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------------------------
// small numeric helpers
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx_ftz(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// the reference's __expf under --use_fast_math: ex2.approx.ftz(x * log2(e))  (moe/gate.cuh:580-583)
__device__ __forceinline__ float fast_expf(float x) { return ex2_approx_ftz(x * 1.4426950408889634f); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);  // RNE, like cutlass::NumericConverter
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_bits_to_f32(uint32_t bits16) { return __uint_as_float(bits16 << 16); }
__device__ __forceinline__ float rne_bf16(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

}  // namespace fm
