// tc_ptx.cuh -- inline-PTX wrappers shared by the tcgen05 kernels (sm_100a): mbarriers, TMA loads / stores,
// tcgen05 alloc / mma / commit / ld, UMMA shared-memory and instruction descriptors.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace {

constexpr int BLOCK_M = 128;
constexpr int kRowBytes = 128;  // one swizzle row per pixel per K-step: 32 fp32 (kind::tf32, K=8 per MMA)
                                // or 64 fp16 (kind::f16, K=16 per MMA); four MMAs per K-step either way

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* smem, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint64_t* bar, void* smem, int c0, int c1,
                                            int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) (ignored for swizzled K-major, 1) | SBO>>4 [32,46) = 8 rows * 128 B
// | version=1 [46,48) | layout SWIZZLE_128B = 2 [61,64)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// M/N-major, 128-byte swizzle descriptor (the operand is stored with M or N contiguous): one swizzle atom is 64 M/N
// elements (one 128-byte row) x 8 K rows (1024 B).  Here SBO is the step between 8-row K groups (1024 B: the K rows of
// a TMA box follow each other) and LBO the step between 64-element M/N blocks (`mn_block_bytes`: one TMA box each).
// An MMA with K = 16 reads two K groups; the next one starts 2048 B further on.
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr, uint32_t mn_block_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(mn_block_bytes >> 4) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 (1<<4), A=TF32 (2<<7),
// B=TF32 (2<<10), A/B K-major (bits 15/16 = 0), N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int n, bool f16) {
    return (1u << 4) | ((f16 ? 0u : 2u) << 7) | ((f16 ? 0u : 2u) << 10) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(BLOCK_M >> 4) << 24);
}
// the same with the transpose bits: A (bit 15) and / or B (bit 16) read M/N-major from shared memory
__host__ __device__ constexpr uint32_t make_idesc_major(int n, bool f16, bool a_mn, bool b_mn) {
    return make_idesc(n, f16) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32"
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
        " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void sts128(uint32_t saddr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts128u(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds128u(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
    return v;
}
// bring `bytes` (multiple of 16, 16-byte aligned) of global memory into L2 ahead of use; no registers, no smem
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n"
        ".reg .pred P;\n"
        "elect.sync _|P, 0xffffffff;\n"
        "selp.b32 %0, 1, 0, P;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---- CTA pairs (cta_group::2): cluster rank, cluster barrier, remote mbarrier arrive, 2-SM MMA / commit / alloc
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory variable in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa_rank(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// wait with cluster-scope acquire (the arrival came from the peer CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAITC:\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONEC;\n"
        "bra LAB_WAITC;\n"
        "DONEC:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
        : "memory");
}
// the barrier at this offset in BOTH CTAs of the pair receives one arrival when the pair's MMAs retire
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}
// TMA loads of a CTA pair: data lands in the executing CTA's shared memory, the completion is signalled on a barrier
// that may live in EITHER CTA of the pair (bar_cluster_addr: a shared::cluster address, e.g. mapa_rank(.., 0))
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint32_t bar_cluster_addr, void* smem, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(const CUtensorMap* map, uint32_t bar_cluster_addr, void* smem, int c0, int c1,
                                                 int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
        : "memory");
}
// instruction descriptor of the pair's MMA: M = 256 (128 rows per CTA)
__host__ __device__ constexpr uint32_t make_idesc_2cta(int n, bool f16) {
    return (1u << 4) | ((f16 ? 0u : 2u) << 7) | ((f16 ? 0u : 2u) << 10) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(256 >> 4) << 24);
}

// ---- TMA stores (shared -> global through a tensor map, bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_wait_group_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_wait_group() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

}  // namespace
