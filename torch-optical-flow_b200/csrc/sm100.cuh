// sm100.cuh -- the Blackwell async layer shared by the TMA / tcgen05 kernels (corr_gemm.cu, gemm_bf16.cu, warp_tma.cu):
// mbarriers, TMA tensor loads, tcgen05 MMA and TMEM access as inline PTX, and the host's tensor-map encoder.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace ofb {

// ------------------------------------------------------------------------------------ mbarriers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(bar), "r"(rank) : "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
constexpr uint32_t MBAR_MAX_POLLS = 1u << 26;   // far above the longest legitimate wait (a long-K backward tile's epilogue)
// Bounded wait: a protocol bug becomes a trapped launch, never a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > MBAR_MAX_POLLS) __trap();
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// ------------------------------------------------------------------------------------ fences and clusters
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}

// ------------------------------------------------------------------------------------ TMA loads
// The completion bytes are credited to `bar` (a shared::cluster address: for a CTA pair the leader's barrier collects
// both CTAs' loads).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
template <int CG>
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            uint64_t pol) {
    if (CG == 1)
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
            ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(pol) : "memory");
    else
        asm volatile(
            "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
            ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(pol) : "memory");
}
// without an L2 hint
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
template <int CG>
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3, uint64_t pol) {
    if (CG == 1)
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
            ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol) : "memory");
    else
        asm volatile(
            "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
            ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol) : "memory");
}
// The same box delivered to the SAME CTA-relative offset (data and mbarrier) of every CTA in `mask`: one L2 read
// feeds both CTAs of a cluster.
__device__ __forceinline__ void tma_load_4d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                               int c3, uint16_t mask, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint "
        "[%0], [%1, {%3, %4, %5, %6}], [%2], %7, %8;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(mask), "l"(pol) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}

// ------------------------------------------------------------------------------------ tcgen05 / TMEM
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    if (CG == 1) asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    else         asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_relinquish() {
    if (CG == 1) asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    else         asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
    else         asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (CG == 1)
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when they retire (both CTAs of a pair)
template <int CG>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if (CG == 1)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    else
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
            ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// cta_group::1 MMAs retiring -> one arrival on the barrier at this offset in BOTH CTAs of the cluster
__device__ __forceinline__ void umma_commit_both(uint32_t bar) {
    asm volatile(
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// 32 lanes x 64 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&v)[64]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
        "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
        "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]),
          "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]),
          "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]),
          "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]),
          "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
        : "r"(taddr) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart
// (cute::UMMA::SmemDescriptor: start >> 4 | LBO [16,30) | SBO [32,46) | version=1 [46,48) | layout [61,64))
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;                 // leading byte offset: unused for swizzled K-major, canonical value 1
    d |= (uint64_t)(1024 >> 4) << 32;       // stride byte offset: 8 rows x 128 B
    d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
    return d;
}
// kind::f16 operand formats (the a_format [7,10) and b_format [10,13) fields of the instruction descriptor)
constexpr uint32_t UMMA_F16 = 0, UMMA_BF16 = 1;
// kind::f16 instruction descriptor: D fp32, A = B = `ab_format` (bf16 by default), both K-major
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, uint32_t ab_format = UMMA_BF16) {
    return (1u << 4) | (ab_format << 7) | (ab_format << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// The 16-bit operand / storage type T as the tcgen05 and TMA descriptors name it
template <typename T> struct F16Format;
template <> struct F16Format<__nv_bfloat16> {
    static constexpr uint32_t umma = UMMA_BF16;
    static constexpr CUtensorMapDataType tma = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
};
template <> struct F16Format<__half> {
    static constexpr uint32_t umma = UMMA_F16;
    static constexpr CUtensorMapDataType tma = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
};

// ------------------------------------------------------------------------------------ host side
// cuTensorMapEncodeTiled with no interleave and no out-of-bounds NaN fill (TMA zero-fills outside the tensor).
// dims, box: `rank` entries, innermost first; strides_bytes: the rank - 1 outer strides.  False when the driver
// entry point is missing or rejects the map.  Defined in api.cu.
bool encode_tiled(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims,
                  const cuuint64_t* strides_bytes, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                  CUtensorMapL2promotion l2_promotion);

}  // namespace ofb
