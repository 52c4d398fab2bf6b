// corr_gemm.cu -- K2: all-pairs correlation pyramid on the 5th-generation tensor cores (version 2).
//
// Replaces CorrBlock.corr + CorrBlock.__init__ (reference methods/raft/model/corr.py:38-54,79-87):
//     corr[b,p,q] = sum_c f1[b,c,p] * f2[b,c,q] / sqrt(C)          (torch.matmul + full-volume divide)
//     level l     = 2x2 average pooling of level l-1 over the target image, complete blocks only
// The reference makes one cuBLAS launch plus 4 further full passes over a multi-GB volume.  Here one
// persistent kernel produces a level AND its 2x2-pooled successor straight from the accumulators; it
// runs twice: on fmap2 (levels 0, 1) and on the 4x4-averaged fmap2 (levels 2, 3) -- pooling is linear,
// avgpool4(f1^T f2) = f1^T avgpool4(f2), and the second run costs 1/16 of the first.
//
//   * operands are K-major bf16 (ofb_corr_prep_bf16: cast + transpose, 1/sqrt(C) folded into fmap1) or fp16
//     (ofb_corr_prep_to; the scale is applied to the accumulators, the reference's order under autocast),
//     fetched by TMA with 128-byte swizzle.  The storage type T is a template parameter: it reaches only the
//     instruction descriptor, the tensor maps and the epilogue's pack instruction;
//   * a CTA owns 128 queries (rows of the volume): their 128 x C slice of fmap1 stays RESIDENT in
//     shared memory while the CTA walks target tiles; only fmap2 streams through a 96..160 KiB TMA ring;
//   * a target tile is 256 targets laid out as 4 "chunks" of 2 rows x 32 columns of the target image
//     (tile shape 32x8, 64x4 or 128x2, whichever wastes least for the image width), fetched as 4-D TMA
//     boxes (C, x, y, b).  TMA zero-fills outside the image;
//   * tcgen05.mma (kind::f16, bf16 x bf16 or fp16 x fp16 -> fp32) accumulates 128 x 256 in TMEM, two accumulator
//     stages (2 x 256 of the 512 columns) so the epilogue of tile n overlaps the MMAs of tile n+1;
//   * cta_group = 2: a CTA PAIR shares each target tile (each CTA loads half of it, the MMA is M = 256
//     across the pair) -- halves the L2 -> SM operand traffic, which is what bounds cta_group = 1
//     (measured: 37 B/cycle/SM, profiles/r01_k2_findings.md);
//   * epilogue: 8 warps; a thread owns one query row and one 64-column chunk at a time
//     (tcgen05.ld 32x32b.x64).  A chunk is a pool-closed patch of the target image (16 x 4 for the 8x4-blocked
//     layouts, 32 x 2 for rows), so the 2x2 means are sums of registers of ONE thread.  Output leaves through
//     the LSU, not TMA (TMA tensor stores cost ~5 cycles per box row and these rows are 64 bytes):
//       - query-minor blocked layout (default): the lane's two 64-byte block slots are its own and the 32 lanes'
//         slots are adjacent, so every lane stores full 32-byte sectors straight from registers
//         (st.global.v8.b32) -- no shared-memory transpose, no barriers; a warp fills 2 KiB runs;
//       - query-major layouts: each warp transposes its 32 x 128 B through a private XOR-swizzled
//         shared-memory stage and writes 16-byte pieces, 8 lanes per 128-byte run.
//
// Roofline (DESIGN.md section 4): 2*B*N^2*C flops against the bf16 tensor peak and 2 bytes * 1.33 *
// B*N^2 of pyramid writes against HBM; at C = 256 and 1965 MHz the write is the larger bound.
#include <cstdlib>
#include <type_traits>

#include "sm100.cuh"

namespace {

using namespace ofb;

constexpr int BLOCK_M = 128;
constexpr int TILE_N = 256;                 // accumulator columns = 4 chunks x (2 rows x 32 cols)
constexpr int CHUNK = 64;
constexpr int BLOCK_K = 64;                 // one 128-byte swizzle span of bf16
constexpr int UMMA_K = 16;
constexpr int MAX_KB = 4;                   // C <= 256
constexpr int A_KB_BYTES = BLOCK_M * BLOCK_K * 2;          // 16 KiB
constexpr int B_TILE_KB_BYTES = TILE_N * BLOCK_K * 2;      // 32 KiB per k-block for a whole tile
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 64 + NUM_EPI_WARPS * 32;       // warp 0: TMA, warp 1: MMA + TMEM, warps 2..9: epilogue
constexpr int TMEM_COLS = 512;
constexpr int MAX_STAGES = 10;
constexpr int PROF_SLOT = 148 * 16;         // uint64 counters per GEMM run in the diagnostics buffer

constexpr int STG_A_BYTES = 32 * 128;       // per warp: 32 queries x (2 rows x 32 bf16)
constexpr int STG_B_BYTES = 32 * 32;        // per warp: 32 queries x 16 bf16 (pooled)
constexpr int STG_WARP_BYTES = STG_A_BYTES + STG_B_BYTES;

constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + MAX_KB * A_KB_BYTES;         // 64 KiB, 1024-aligned
// The query-minor layout needs no epilogue staging (direct register stores): its shared memory goes to a deeper
// operand ring instead (the stream is latency-bound: 2 / 3 stages of 32 KiB measured 6900 / 5000 cycles per tile).
// Epilogue store modes of the query-minor layout:
//   EPI_DIRECT  32-byte register stores (st.global.v8.b32), no staging: the whole budget goes to a 5-stage operand ring;
//   EPI_BULK    each warp stages one 8x4 block of its 32 queries -- 2 KiB that are CONTIGUOUS in the query-minor layout --
//               in shared memory and hands it to the TMA engine (cp.async.bulk.global.shared::cta): full-line writes that
//               never pass through the LSU, and the warp does not wait for them (round-2 probes, DESIGN.md section 4).
//   EPI_PIPE    EPI_DIRECT's stores, software-pipelined: the accumulator leaves TMEM in 32-column pieces (two block rows of
//               two blocks = exactly two 32-byte sector stores per lane), and the tcgen05.ld of piece p+1 -- across tile
//               boundaries too -- is in flight while piece p is converted and stored.  Measured (profiles/r02_k2_ablate*):
//               with 8 warps sharing the TMEM read port a 64-column tcgen05.ld stalls its warp for ~850 cycles, and in
//               EPI_DIRECT that stall and the ~1170 cycles of store issue per chunk are serial.
constexpr int EPI_DIRECT = 0, EPI_BULK = 1, EPI_PIPE = 2;
constexpr int BULK_BLOCK_BYTES = 32 * 64;                      // 32 queries x one 64-byte block slot
constexpr int BULK_WARP_BYTES = 2 * BULK_BLOCK_BYTES;          // X: the level-0 block in flight, Y: the warp's level-1 block
template <int CG, int LAY, int EPI = EPI_DIRECT> struct Ring {
    static constexpr bool STAGED = LAY != OFB_LAYOUT_QMINOR8X4;
    static constexpr bool BULK = !STAGED && EPI == EPI_BULK;
    static constexpr int STAGE_BYTES = B_TILE_KB_BYTES / CG;              // 32 KiB / 16 KiB
    static constexpr int STAGES = (STAGED ? 3 : BULK ? 4 : 5) * CG;       // 96 / 128 / 160 KiB
    static constexpr int OFF_STG = OFF_B + STAGES * STAGE_BYTES;
    static constexpr int OFF_BAR = OFF_STG + (STAGED ? NUM_EPI_WARPS * STG_WARP_BYTES : BULK ? NUM_EPI_WARPS * BULK_WARP_BYTES : 0);
    static constexpr int NUM_BARS = 2 + 2 * MAX_STAGES + 4;                // a_full, a_empty, b_full[], b_empty[], t_full[2], t_empty[2]
    static constexpr int SMEM_BYTES = OFF_BAR + NUM_BARS * 8 + 16;
    static constexpr int SMEM_ALLOC = SMEM_BYTES + 1024;                   // manual 1024-byte alignment of the dynamic segment
};
static_assert(Ring<1, 0>::SMEM_ALLOC <= 232448 && Ring<2, 0>::SMEM_ALLOC <= 232448 && Ring<1, 2>::SMEM_ALLOC <= 232448 &&
              Ring<2, 2>::SMEM_ALLOC <= 232448 && Ring<2, 2>::STAGES <= MAX_STAGES && Ring<1, 2, 1>::SMEM_ALLOC <= 232448 &&
              Ring<2, 2, 1>::SMEM_ALLOC <= 232448, "shared memory budget");

// One level of a run's output, copied from the PyramidView (level_out): fields side by side keep the kernel's code
template <typename T> struct LevelOut {
    T* base;                     // 16-bit storage: __nv_bfloat16 or __half
    long long q_stride;
    int pitch, h, w;
    int blocked;                 // PyramidView::blocked
    long long blk_stride;        // PyramidView::blk_stride
};
template <typename T>
LevelOut<T> level_out(const PyramidView& v, int l) {
    return {static_cast<T*>(v.base[l]), v.q_stride[l], v.pitch[l], v.lh[l], v.lw[l], v.blocked, v.blk_stride};
}
// element offset (without the query term q * q_stride) of the 8-element piece starting at (y, x), x % 8 == 0
template <typename T>
__device__ __forceinline__ long long piece_offset(const LevelOut<T>& L, int y, int x) {
    return OFB_PIECE_OFFSET(L, y, x, L.pitch);
}

template <typename T> struct GemmParams {
    int B, C, kb;
    int Nq;                      // queries per batch element (rows of the volume)
    int th, tw;                  // target image of THIS run (h x w, or h/4 x w/4 for the pooled run)
    int CW, CR;                  // chunk = CW x CR targets (64): 32 x 2 for row layouts, 16 x 4 for 8x4-blocked layouts
    int XB, YQ;                  // tile = XB x YQ chunks (XB * YQ = 4) = (CW*XB) x (CR*YQ) targets
    int nbox, box_rows;          // TMA boxes per stage and CTA, rows per box
    int ntx, nty, ntiles;
    int tiles_per_item, n_chunks, mblk, n_items;
    float scale;
    int apply_scale, has_b;
    LevelOut<T> la, lb;          // level written from the accumulators, and its 2x2 mean
    int dbg;                     // PROF builds only: bit mask disabling parts of the epilogue (tools/k2_profile.py)
    unsigned long long* prof;    // optional per-CTA wait-cycle counters (ofb_corr_pyramid_bf16_profile)
};

// ------------------------------------------------------------------------------------ PTX helpers
template <bool PROF>
__device__ __forceinline__ void mbar_wait_p(uint32_t bar, uint32_t parity, unsigned long long& acc) {
    if (PROF) {
        const long long t0 = clock64();
        mbar_wait(bar, parity);
        acc += (unsigned long long)(clock64() - t0);
    } else {
        mbar_wait(bar, parity);
    }
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
// two fp32 values -> one word of the 16-bit storage type T (round to nearest even)
template <typename T> __device__ __forceinline__ uint32_t pack16(float lo, float hi) {
    if constexpr (std::is_same<T, __half>::value) return pack_f16(lo, hi);
    else return pack_bf16(lo, hi);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr) : "memory");
    return r;
}
// streaming (evict-first) 16-byte store: the volume is written once and must not push fmap2 out of L2
__device__ __forceinline__ void st_global_v4(void* p, uint4 v) {
    asm volatile("st.global.cs.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// 32-byte store (sm_100): one full sector per lane
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t* a, const uint32_t* b) {
    asm volatile("st.global.cs.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(p), "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]) : "memory");
}

// TMA bulk store of a contiguous run, shared -> global; completion is tracked per issuing thread in bulk async-groups
__device__ __forceinline__ void bulk_store(void* gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all of this thread's bulk stores have finished READING shared memory (the staging buffer may be rewritten)
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy writes (st.shared) -> visible to the async proxy (the TMA engine)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// One 64-byte block slot per lane -> the warp's staging buffer, conflict-free: the four 16-byte pieces (block rows) of a
// lane are stored in the order (i + rot) & 3 with rot = (lane >> 1) & 3, so the 8 lanes of a store phase hit 8 different
// 16-byte bank groups although their slots are 64 bytes apart.  The register file cannot be indexed dynamically: the
// pieces are rotated by `rot` with two select stages first.  p0..p3 = the lane's pieces in memory order.
__device__ __forceinline__ void stage_slot(uint32_t slot, uint32_t rot, const uint32_t* p0, const uint32_t* p1,
                                           const uint32_t* p2, const uint32_t* p3) {
    const bool r1 = rot & 1u, r2 = rot & 2u;
    uint32_t a[4][4], b[4][4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        a[0][e] = r1 ? p1[e] : p0[e]; a[1][e] = r1 ? p2[e] : p1[e];
        a[2][e] = r1 ? p3[e] : p2[e]; a[3][e] = r1 ? p0[e] : p3[e];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) b[i][e] = r2 ? a[(i + 2) & 3][e] : a[i][e];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        st_shared_v4(slot + ((((uint32_t)i + rot) & 3u) << 4), b[i][0], b[i][1], b[i][2], b[i][3]);
}

struct ItemCoord {
    int b, chunk, m;
};
template <typename GP>
__device__ __forceinline__ ItemCoord decode_item(const GP& P, int item) {
    ItemCoord ic;
    ic.m = item % P.mblk;
    const int r = item / P.mblk;
    ic.chunk = r % P.n_chunks;
    ic.b = r / P.n_chunks;
    return ic;
}

// The (item, tile) sequence of one worker, as the three roles walk it.
template <typename T> struct TileIter {
    int item, t, t1;
    ItemCoord ic;
    bool valid;
    __device__ __forceinline__ void load(const GemmParams<T>& P) {
        valid = item < P.n_items;
        if (valid) {
            ic = decode_item(P, item);
            t = ic.chunk * P.tiles_per_item;
            t1 = min(t + P.tiles_per_item, P.ntiles);
        }
    }
    __device__ __forceinline__ void init(const GemmParams<T>& P, int worker) { item = worker; load(P); }
    __device__ __forceinline__ void advance(const GemmParams<T>& P, int n_workers) {
        if (++t >= t1) { item += n_workers; load(P); }
    }
};

// EPI_PIPE: one 32-column piece = block rows 2*rh, 2*rh+1 of the chunk's two 8x4 blocks (chunk = 16 x 4 targets, column
// c = row * 16 + x).  Level 0: one 32-byte sector per block.  Level 1: the piece closes ONE pooled row (8 means); the
// even piece keeps it in `keep`, the odd piece stores both rows as one sector.
template <typename T>
__device__ __forceinline__ void store_piece(const GemmParams<T>& P, const uint32_t (&v)[32], int rh, int x0, int y0,
                                            long long qg, bool qok, uint32_t (&keep)[4]) {
    float f[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) f[c] = P.apply_scale ? __uint_as_float(v[c]) * P.scale : __uint_as_float(v[c]);
    if (qok && y0 < P.la.h) {
#pragma unroll
        for (int b2 = 0; b2 < 2; ++b2) {
            const int x = x0 + b2 * 8;
            if (x < P.la.pitch) {
                uint32_t r0[4], r1[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    r0[e] = pack16<T>(f[b2 * 8 + 2 * e], f[b2 * 8 + 2 * e + 1]);
                    r1[e] = pack16<T>(f[16 + b2 * 8 + 2 * e], f[16 + b2 * 8 + 2 * e + 1]);
                }
                st_global_v8(P.la.base + qg * P.la.q_stride + piece_offset(P.la, y0, x) + rh * 16, r0, r1);
            }
        }
    }
    if (P.has_b) {
        uint32_t mk[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {       // 2x2 means, summed in the reference's raster order then / 4 (corr.py:53)
            const int a0 = 4 * e, a1 = 4 * e + 2;
            const float m0 = (((f[a0] + f[a0 + 1]) + f[a0 + 16]) + f[a0 + 17]) * 0.25f;
            const float m1 = (((f[a1] + f[a1 + 1]) + f[a1 + 16]) + f[a1 + 17]) * 0.25f;
            mk[e] = pack16<T>(m0, m1);
        }
        if (rh == 0) {
#pragma unroll
            for (int e = 0; e < 4; ++e) keep[e] = mk[e];
        } else {
            const int y = y0 >> 1, x = x0 >> 1;
            if (qok && y < P.lb.h && x < P.lb.pitch)
                st_global_v8(P.lb.base + qg * P.lb.q_stride + piece_offset(P.lb, y, x), keep, mk);
        }
    }
}

// ------------------------------------------------------------------------------------ the kernel
// LAY: output layout (OFB_LAYOUT_ROWS / BLOCK8X4 / QMINOR8X4)
// T: 16-bit operand and pyramid storage type (__nv_bfloat16 or __half)
// MC (CG == 1 only): CTAs run as CLUSTERS OF TWO that walk the same target tiles with their own 128 queries each, their own
// accumulators and their own cta_group::1 MMAs; every fmap2 stage is fetched half by each CTA and MULTICAST into both, so
// the L2 -> SM operand stream is halved (as with cta_group::2) while the two epilogues stay independent.
template <typename T, int CG, bool PROF, int LAY, int EPI, bool MC>
__global__ void __launch_bounds__(NUM_THREADS, 1)
corr_pyramid_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const GemmParams<T> P) {
    static_assert(!MC || CG == 1, "multicast clusters issue cta_group::1 MMAs");
    using R = Ring<CG, LAY, EPI>;
    constexpr bool BULK = R::BULK;
    constexpr int CL = (CG == 2 || MC) ? 2 : 1;                  // CTAs per cluster
    constexpr bool BLK = LAY != OFB_LAYOUT_ROWS;
    extern __shared__ uint8_t smem_raw[];
    // the 128-byte swizzle is a function of the absolute shared address: align the segment to 1024
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - raw);
    constexpr int B_STAGE_BYTES = R::STAGE_BYTES;
    constexpr int B_STAGES = R::STAGES;

    const uint32_t bar0 = sbase + R::OFF_BAR;
    const uint32_t bar_a_full = bar0, bar_a_empty = bar0 + 8;
    const uint32_t bar_b_full = bar0 + 16, bar_b_empty = bar0 + 16 + 8 * MAX_STAGES;
    const uint32_t bar_t_full = bar0 + 16 + 16 * MAX_STAGES, bar_t_empty = bar_t_full + 16;
    const uint32_t tmem_slot = bar0 + R::NUM_BARS * 8;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(sgen + R::OFF_BAR + R::NUM_BARS * 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = (CL == 2) ? cluster_ctarank() : 0u;
    const bool leader = rank == 0;
    const int worker = blockIdx.x / CL, n_workers = gridDim.x / CL;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_a); prefetch_tmap(&map_b);
        mbar_init(bar_a_full, 1);
        mbar_init(bar_a_empty, 1);
        // multicast: a stage is written in BOTH CTAs by either producer, so it is free when both MMA lanes are done with it
        for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(bar_b_full + 8 * s, 1); mbar_init(bar_b_empty + 8 * s, MC ? 2 : 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(bar_t_full + 8 * s, 1); mbar_init(bar_t_empty + 8 * s, NUM_EPI_WARPS * CG); }
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc<CG>(tmem_slot, TMEM_COLS);
        tmem_relinquish<CG>();
    }
    tc_fence_before();
    if (CL == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    const int m_rows = BLOCK_M * CL;   // query rows per work item
    const long long t_start = PROF ? clock64() : 0;
    const int dbg = PROF ? P.dbg : 0;
    unsigned long long pw0 = 0, pw1 = 0, pw2 = 0, ptiles = 0;   // per-role wait cycles (PROF only)
    unsigned long long p_ld = 0, p_st = 0, p_bw = 0;            // epilogue: tcgen05.ld + wait, store section, bulk-wait

    if (warp == 0) {
        // ============================== TMA producer (one lane) ==============================
        if (lane == 0) {
            const uint32_t full_a = (CG == 2) ? map_to_rank(bar_a_full, 0) : bar_a_full;
            // which part of the tile this CTA fetches (cta_group 2: chunks {2*rank, 2*rank+1})
            const int TH = P.CR * P.YQ;
            const int xb0 = (CL == 2 && P.XB >= 2) ? (int)rank * (P.XB / 2) : 0;
            const int yoff = (CL == 2 && P.XB == 1) ? (int)rank * (TH / 2) : 0;
            const int box_bytes = P.CW * P.box_rows * 128;
            // the operands are re-read by every CTA: keep them in L2 (evict_last) against the streaming pyramid writes
            const uint64_t pol = l2_policy_evict_last();
            uint32_t stage = 0, bphase = 0, aphase = 0;
            for (int item = worker; item < P.n_items; item += n_workers) {
                const ItemCoord ic = decode_item(P, item);
                mbar_wait_p<PROF>(bar_a_empty, aphase ^ 1, pw1);
                aphase ^= 1;
                if (leader || MC) mbar_expect_tx(bar_a_full, (uint32_t)(P.kb * A_KB_BYTES * CG));
                const int row0 = ic.m * m_rows + (int)rank * BLOCK_M;
                for (int kb = 0; kb < P.kb; ++kb)
                    tma_load_3d<CG>(sbase + OFF_A + kb * A_KB_BYTES, &map_a, full_a, kb * BLOCK_K, row0, ic.b, pol);
                const int t0 = ic.chunk * P.tiles_per_item;
                const int t1 = min(t0 + P.tiles_per_item, P.ntiles);
                for (int t = t0; t < t1; ++t) {
                    const int ty = t / P.ntx, tx = t - ty * P.ntx;
                    const int x0 = (tx * P.XB + xb0) * P.CW, y0 = ty * TH + yoff;
                    for (int kb = 0; kb < P.kb; ++kb) {
                        mbar_wait_p<PROF>(bar_b_empty + 8 * stage, bphase ^ 1, pw0);
                        const uint32_t full_b = (CG == 2) ? map_to_rank(bar_b_full + 8 * stage, 0) : bar_b_full + 8 * stage;
                        if (leader || MC) mbar_expect_tx(bar_b_full + 8 * stage, (uint32_t)B_TILE_KB_BYTES);
                        // multicast: this CTA's half of the tile goes to the same place in both CTAs
                        const uint32_t dst = sbase + OFF_B + stage * B_STAGE_BYTES + (MC ? rank * (uint32_t)(B_TILE_KB_BYTES / 2) : 0u);
                        for (int j = 0; j < P.nbox; ++j) {
                            if (MC) tma_load_4d_mc(dst + j * box_bytes, &map_b, full_b, kb * BLOCK_K, x0 + P.CW * j, y0, ic.b, (uint16_t)3, pol);
                            else tma_load_4d<CG>(dst + j * box_bytes, &map_b, full_b, kb * BLOCK_K, x0 + P.CW * j, y0, ic.b, pol);
                        }
                        if (++stage == B_STAGES) { stage = 0; bphase ^= 1; }
                    }
                }
            }
            if (PROF && P.prof) {
                unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
                o[0] = pw0; o[1] = pw1;
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ============================== MMA issuer (leader CTA, one lane) ====================
        if ((leader || MC) && lane == 0) {
            constexpr uint32_t idesc = make_idesc(BLOCK_M * CG, TILE_N, F16Format<T>::umma);
            uint32_t stage = 0, bphase = 0, aphase = 0, acc = 0, tphase = 0;
            for (int item = worker; item < P.n_items; item += n_workers) {
                const ItemCoord ic = decode_item(P, item);
                mbar_wait_p<PROF>(bar_a_full, aphase, pw0);
                aphase ^= 1;
                tc_fence_after();
                const int t0 = ic.chunk * P.tiles_per_item;
                const int t1 = min(t0 + P.tiles_per_item, P.ntiles);
                for (int t = t0; t < t1; ++t) {
                    mbar_wait_p<PROF>(bar_t_empty + 8 * acc, tphase ^ 1, pw1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * TILE_N;
                    for (int kb = 0; kb < P.kb; ++kb) {
                        mbar_wait_p<PROF>(bar_b_full + 8 * stage, bphase, pw2);
                        tc_fence_after();
                        const uint64_t adesc = make_smem_desc(sbase + OFF_A + kb * A_KB_BYTES);
                        const uint64_t bdesc = make_smem_desc(sbase + OFF_B + stage * B_STAGE_BYTES);
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                            // advance both start addresses by k * 16 elements * 2 B = 32 B (>> 4 = 2)
                            umma_bf16<CG>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc,
                                          (uint32_t)((kb | k) != 0));
                        }
                        if (MC) umma_commit_both(bar_b_empty + 8 * stage);   // both CTAs' producers may refill it
                        else umma_commit<CG>(bar_b_empty + 8 * stage); // smem stage free once these MMAs retire
                        if (++stage == B_STAGES) { stage = 0; bphase ^= 1; }
                    }
                    umma_commit<CG>(bar_t_full + 8 * acc);             // accumulator ready for the epilogue
                    if (++acc == 2) { acc = 0; tphase ^= 1; }
                }
                umma_commit<CG>(bar_a_empty);                          // resident A may be replaced
            }
            if (PROF && P.prof) {
                unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
                o[2] = pw0; o[3] = pw1; o[4] = pw2;
            }
        }
        __syncwarp();
    } else if (EPI == EPI_PIPE && LAY == OFB_LAYOUT_QMINOR8X4) {
        // ============================== epilogue, software-pipelined (8 warps) ===============
        const int q4 = warp & 3, half = (warp - 2) >> 2;
        uint32_t acc = 0, tphase = 0;
        TileIter<T> it;
        it.init(P, worker);
        if (it.valid) {
            uint32_t buf0[32], buf1[32], keep[4] = {0, 0, 0, 0};
            const uint32_t tlane = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)half * 2 * CHUNK;
            mbar_wait_p<PROF>(bar_t_full + 8 * acc, tphase, pw0);
            tc_fence_after();
            uint32_t taddr = tlane + acc * TILE_N;
            tmem_ld32(taddr, buf0);
            while (true) {
                if (PROF) ++ptiles;
                const int ty = it.t / P.ntx, tx = it.t - ty * P.ntx;
                const int qrow = it.ic.m * m_rows + (int)rank * BLOCK_M + q4 * 32 + lane;     // this lane's query row
                const bool qok = qrow < P.Nq;
                const long long qg = (long long)it.ic.b * P.Nq + qrow;
                TileIter<T> nxt = it;
                nxt.advance(P, n_workers);
                uint32_t taddr_next = 0;
#pragma unroll
                for (int pc = 0; pc < 4; ++pc) {
                    tmem_ld_wait();                                   // piece pc has landed (the only load in flight)
                    if (pc < 3) {
                        if ((pc & 1) == 0) tmem_ld32(taddr + (pc + 1) * 32, buf1);
                        else tmem_ld32(taddr + (pc + 1) * 32, buf0);
                    } else {
                        // all four pieces of this warp have left TMEM: hand the accumulator stage back ...
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (CG == 2) mbar_arrive_cluster(bar_t_empty + 8 * acc, 0);
                            else mbar_arrive(bar_t_empty + 8 * acc);
                        }
                        if (++acc == 2) { acc = 0; tphase ^= 1; }
                        // ... and fetch the first piece of the next tile before this tile's last stores are issued
                        if (nxt.valid) {
                            mbar_wait_p<PROF>(bar_t_full + 8 * acc, tphase, pw0);
                            tc_fence_after();
                            taddr_next = tlane + acc * TILE_N;
                            tmem_ld32(taddr_next, buf0);
                        }
                    }
                    const int k = half * 2 + (pc >> 1);
                    const int xb = k / P.YQ, yq = k - xb * P.YQ;
                    const int x0 = (tx * P.XB + xb) * P.CW, y0 = (ty * P.YQ + yq) * P.CR;
                    if (!(PROF && (dbg & 1))) {
                        if ((pc & 1) == 0) store_piece(P, buf0, 0, x0, y0, qg, qok, keep);
                        else store_piece(P, buf1, 1, x0, y0, qg, qok, keep);
                    }
                }
                if (!nxt.valid) break;
                it = nxt;
                taddr = taddr_next;
            }
        }
        if (PROF && P.prof && warp == 2 && lane == 0) {
            unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
            o[5] = pw0; o[6] = 0; o[7] = ptiles; o[8] = (unsigned long long)(clock64() - t_start);
        }
    } else {
        // ============================== epilogue (8 warps) ===================================
        // warp -> TMEM lane quarter (hardware rule: warp_id % 4) and column half; thread -> one query row
        const int q4 = warp & 3;
        const int half = (warp - 2) >> 2;
        const uint32_t stg_a = sbase + R::OFF_STG + (warp - 2) * STG_WARP_BYTES;
        const uint32_t stg_b = stg_a + STG_A_BYTES;
        // write side of the transposes: this lane's query row, 16-byte pieces XOR-swizzled
        const uint32_t wa = stg_a + (uint32_t)lane * 128u, wsw_a = (uint32_t)(lane & 7);
        const uint32_t wb = stg_b + (uint32_t)lane * 32u, wsw_b = (uint32_t)((lane >> 2) & 1);
        // read side: level A -- 8 lanes per query, 4 queries per instruction.  Lanes follow MEMORY order:
        // rows: piece p = (row p>>2, columns 8*(p&3));  8x4 blocks: memory piece m = (block m>>2, block row m&3)
        // is register piece p = (row p>>1, block p&1) -- the chunk's two blocks are one contiguous 128-byte line
        const int ra_q = lane >> 3;
        const int ra_p = BLK ? ((((lane & 7) & 3) << 1) | ((lane & 7) >> 2)) : (lane & 7);
        const int ra_dy = BLK ? (ra_p >> 1) : (ra_p >> 2), ra_dx = BLK ? (ra_p & 1) * 8 : (ra_p & 3) * 8;
        // query-minor blocks: one block of 8 consecutive queries per instruction (512 contiguous bytes):
        // lane = (query lane>>2, block row lane&3)
        constexpr bool qminor = LAY == OFB_LAYOUT_QMINOR8X4;
        const int qm_q = lane >> 2, qm_s = lane & 3;
        // level B -- 2 lanes per query, 16 queries per instruction
        const int rb_q = lane >> 1, rb_p = lane & 1;
        // bulk-store staging (EPI_BULK): X = the level-0 block in flight, Y = the level-1 block of the tile
        const uint32_t xbuf = sbase + R::OFF_STG + (uint32_t)(warp - 2) * BULK_WARP_BYTES, ybuf = xbuf + BULK_BLOCK_BYTES;
        const uint32_t rot = (uint32_t)(lane >> 1) & 3u;
        const bool bulk_b = P.YQ == 2;          // the warp's two chunks stack vertically: they close one level-1 block
        uint32_t mk_top[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        uint32_t acc = 0, tphase = 0;
        for (int item = worker; item < P.n_items; item += n_workers) {
            const ItemCoord ic = decode_item(P, item);
            const int qrow0 = ic.m * m_rows + (int)rank * BLOCK_M + q4 * 32;   // first query row of this warp
            const long long qglob0 = (long long)ic.b * P.Nq + qrow0;
            const int t0 = ic.chunk * P.tiles_per_item;
            const int t1 = min(t0 + P.tiles_per_item, P.ntiles);
            for (int t = t0; t < t1; ++t) {
                const int ty = t / P.ntx, tx = t - ty * P.ntx;
                mbar_wait_p<PROF>(bar_t_full + 8 * acc, tphase, pw0);
                tc_fence_after();
                if (PROF) ++ptiles;
                const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * TILE_N + (uint32_t)half * 2 * CHUNK;
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) {
                    const int k = half * 2 + cc;
                    uint32_t v[64];
                    if (PROF && (dbg & 32)) {
#pragma unroll
                        for (int c = 0; c < 64; ++c) v[c] = 0x3f800000u + c;
                    } else {
                        const long long tl0 = PROF ? clock64() : 0;
                        tmem_ld64(taddr + cc * CHUNK, v);
                        tmem_ld_wait();
                        if (PROF) p_ld += (unsigned long long)(clock64() - tl0);
                    }
                    if (cc == 1) {
                        // both chunks of this warp have left TMEM: hand the accumulator stage back
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (CG == 2) mbar_arrive_cluster(bar_t_empty + 8 * acc, 0);
                            else mbar_arrive(bar_t_empty + 8 * acc);
                        }
                    }
                    float f[64];
                    if (P.apply_scale) {
#pragma unroll
                        for (int c = 0; c < 64; ++c) f[c] = __uint_as_float(v[c]) * P.scale;
                    } else {
#pragma unroll
                        for (int c = 0; c < 64; ++c) f[c] = __uint_as_float(v[c]);
                    }
                    if (qminor && !(PROF && (dbg & 64))) {
                        // ---- query-minor blocks: a lane's 64-byte block slots are its own and the 32 lanes' slots are
                        // adjacent, so one block of the warp's 32 queries is a contiguous 2 KiB run
                        const int xb = k / P.YQ, yq = k - xb * P.YQ;
                        const int x0 = (tx * P.XB + xb) * P.CW, y0 = (ty * P.YQ + yq) * P.CR;
                        uint32_t pk[32];
#pragma unroll
                        for (int c = 0; c < 32; ++c) pk[c] = pack16<T>(f[2 * c], f[2 * c + 1]);
                        const bool qok = qrow0 + lane < P.Nq;
                        const int nvalid = min(32, P.Nq - qrow0);          // queries of this warp inside the batch element
                        const long long ts0 = PROF ? clock64() : 0;
                        if (!(PROF && (dbg & 1))) {
#pragma unroll
                            for (int b2 = 0; b2 < 2; ++b2) {
                                const int x = x0 + b2 * 8;
                                // register piece (block row yy, block b2) = pk[4 * (2 * yy + b2) ..]
                                if (BULK) {
                                    if (nvalid > 0 && y0 < P.la.h && x < P.la.pitch) {      // warp-uniform
                                        const long long tb0 = PROF ? clock64() : 0;
                                        if (lane == 0) bulk_wait_read_all();               // the previous block has left X
                                        __syncwarp();
                                        if (PROF) p_bw += (unsigned long long)(clock64() - tb0);
                                        stage_slot(xbuf + (uint32_t)lane * 64u, rot, pk + 4 * b2, pk + 4 * (2 + b2),
                                                   pk + 4 * (4 + b2), pk + 4 * (6 + b2));
                                        fence_async_smem();
                                        __syncwarp();
                                        if (lane == 0) {
                                            bulk_store(P.la.base + qglob0 * P.la.q_stride + piece_offset(P.la, y0, x), xbuf,
                                                       (uint32_t)nvalid * 64u);
                                            bulk_commit();
                                        }
                                    }
                                } else if (qok && y0 < P.la.h && x < P.la.pitch) {
                                    // direct: one full 32-byte sector (two block rows) per lane and instruction
                                    T* dst = P.la.base + (qglob0 + lane) * P.la.q_stride + piece_offset(P.la, y0, x);
                                    st_global_v8(dst, pk + 4 * b2, pk + 4 * (2 + b2));
                                    st_global_v8(dst + 16, pk + 4 * (4 + b2), pk + 4 * (6 + b2));
                                }
                            }
                        }
                        if (P.has_b && !(PROF && (dbg & 2))) {
                            uint32_t mk[8];
#pragma unroll
                            for (int c = 0; c < 8; ++c) {       // pooled 2 rows x 8 columns: 2x2 means in raster order / 4
                                const int a0 = ((2 * c) >> 3) * 32 + ((2 * c) & 7) * 2, a1 = ((2 * c + 1) >> 3) * 32 + ((2 * c + 1) & 7) * 2;
                                const float m0 = (((f[a0] + f[a0 + 1]) + f[a0 + 16]) + f[a0 + 17]) * 0.25f;
                                const float m1 = (((f[a1] + f[a1 + 1]) + f[a1 + 16]) + f[a1 + 17]) * 0.25f;
                                mk[c] = pack16<T>(m0, m1);
                            }
                            const int y = y0 >> 1, x = x0 >> 1;
                            if (BULK && bulk_b) {
                                // 2 x 2 chunks per tile: this warp's two chunks are rows 0-1 and rows 2-3 of ONE level-1 block
                                if (cc == 0) {
#pragma unroll
                                    for (int c = 0; c < 8; ++c) mk_top[c] = mk[c];
                                } else if (nvalid > 0 && (y & ~3) < P.lb.h && x < P.lb.pitch) {
                                    if (lane == 0) bulk_wait_read_all();
                                    __syncwarp();
                                    stage_slot(ybuf + (uint32_t)lane * 64u, rot, mk_top, mk_top + 4, mk, mk + 4);
                                    fence_async_smem();
                                    __syncwarp();
                                    if (lane == 0) {
                                        bulk_store(P.lb.base + qglob0 * P.lb.q_stride + piece_offset(P.lb, y & ~3, x), ybuf,
                                                   (uint32_t)nvalid * 64u);
                                        bulk_commit();
                                    }
                                }
                            } else if (qok && y < P.lb.h && x < P.lb.pitch) {
                                st_global_v8(P.lb.base + (qglob0 + lane) * P.lb.q_stride + piece_offset(P.lb, y, x), mk, mk + 4);
                            }
                        }
                        if (PROF) p_st += (unsigned long long)(clock64() - ts0);
                        continue;
                    }
                    // ---- registers -> swizzled stage.  chunk = 2 image rows x 32 columns, piece p = 8 bf16
                    if (!(PROF && (dbg & 16))) {
#pragma unroll
                        for (int p = 0; p < 8; ++p) {
                            const float* s = f + p * 8;
                            st_shared_v4(wa + ((p ^ wsw_a) << 4), pack16<T>(s[0], s[1]), pack16<T>(s[2], s[3]),
                                         pack16<T>(s[4], s[5]), pack16<T>(s[6], s[7]));
                        }
                        if (P.has_b) {
                            // 2x2 means, summed in the reference's raster order then / 4 (corr.py:53)
                            float m[16];
#pragma unroll
                            for (int c = 0; c < 16; ++c) {
                                // row layouts: chunk 2 x 32 -> one pooled row of 16; blocked: chunk 4 x 16 -> 2 rows of 8
                                const int a = BLK ? ((c >> 3) * 32 + (c & 7) * 2) : 2 * c, dn = BLK ? 16 : 32;
                                m[c] = (((f[a] + f[a + 1]) + f[a + dn]) + f[a + dn + 1]) * 0.25f;
                            }
#pragma unroll
                            for (int p = 0; p < 2; ++p) {
                                const float* s = m + p * 8;
                                st_shared_v4(wb + ((p ^ wsw_b) << 4), pack16<T>(s[0], s[1]), pack16<T>(s[2], s[3]),
                                             pack16<T>(s[4], s[5]), pack16<T>(s[6], s[7]));
                            }
                        }
                    }
                    __syncwarp();
                    // ---- stage -> global, 16-byte pieces, 64-byte segments per (query, image row)
                    const int xb = k / P.YQ, yq = k - xb * P.YQ;
                    const int x0 = (tx * P.XB + xb) * P.CW, y0 = (ty * P.YQ + yq) * P.CR;
                    if (!(PROF && (dbg & 1))) {
                        // pieces are always written whole and the row padding (w..pitch) is written too: TMA
                        // zero-fills targets outside the image, so the padding receives zeros (finite values --
                        // the lookup kernel relies on that) and no 32-byte sector is left partially written
                        // (partial sectors measured a 2x slowdown of the whole kernel at w = 156)
                        uint4 val[8];
                        if (qminor) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int r = (j & 3) * 8 + qm_q, p = (qm_s << 1) | (j >> 2);
                                val[j] = ld_shared_v4(stg_a + (uint32_t)r * 128u + (uint32_t)((p ^ (r & 7)) << 4));
                            }
                            const int y = y0 + qm_s;
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int r = (j & 3) * 8 + qm_q, x = x0 + (j >> 2) * 8;
                                if (y < P.la.h && x < P.la.pitch && qrow0 + r < P.Nq)
                                    st_global_v4(P.la.base + (qglob0 + r) * P.la.q_stride + piece_offset(P.la, y, x), val[j]);
                            }
                        } else {
                            const int y = y0 + ra_dy, x = x0 + ra_dx;
                            const bool in_img = y < P.la.h && x < P.la.pitch;
                            const long long off_yx = piece_offset(P.la, y, x);
                            // all 8 shared loads first, then the 8 global stores: the stores do not wait on each other's data
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int r = j * 4 + ra_q;
                                val[j] = ld_shared_v4(stg_a + (uint32_t)r * 128u + (uint32_t)((ra_p ^ (r & 7)) << 4));
                            }
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int r = j * 4 + ra_q;
                                if (in_img && qrow0 + r < P.Nq)
                                    st_global_v4(P.la.base + (qglob0 + r) * P.la.q_stride + off_yx, val[j]);
                            }
                        }
                    }
                    if (P.has_b && !(PROF && (dbg & 2))) {
                        // pooled chunk: rows layout 1 x 16 (pieces side by side); blocked 2 x 8 (pieces = 2 block rows)
                        const int y = (y0 >> 1) + (BLK ? rb_p : 0), x = (x0 >> 1) + (BLK ? 0 : rb_p * 8);
                        const bool in_img = y < P.lb.h && x < P.lb.pitch;
                        const long long off_yx = piece_offset(P.lb, y, x);
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const int r = j * 16 + rb_q;
                            const uint4 val = ld_shared_v4(stg_b + (uint32_t)r * 32u + (uint32_t)((rb_p ^ ((r >> 2) & 1)) << 4));
                            if (in_img && qrow0 + r < P.Nq) {
                                st_global_v4(P.lb.base + (qglob0 + r) * P.lb.q_stride + off_yx, val);
                            }
                        }
                    }
                    __syncwarp();      // the stage is rewritten by the next chunk
                }
                if (++acc == 2) { acc = 0; tphase ^= 1; }
            }
        }
        if (BULK && lane == 0) bulk_wait_all();          // the staging memory and the stores outlive the loop
        if (PROF && P.prof && warp == 2 && lane == 0) {
            unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
            o[5] = pw0; o[6] = p_st; o[7] = ptiles; o[8] = (unsigned long long)(clock64() - t_start);
            o[9] = p_ld; o[10] = p_bw;
        }
    }

    // teardown: nobody may leave (or free TMEM) while a peer can still signal / read this CTA
    tc_fence_before();
    if (CL == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) tmem_dealloc<CG>(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------ host side
template <typename T, int CG, bool PROF, int LAY, int EPI, bool MC>
int launch_gemm(const CUtensorMap& ma, const CUtensorMap& mb, const GemmParams<T>& P, int grid, cudaStream_t st) {
    OFB_CUDA(ofb_smem_once<corr_pyramid_kernel<T, CG, PROF, LAY, EPI, MC>>(Ring<CG, LAY, EPI>::SMEM_ALLOC));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = Ring<CG, LAY, EPI>::SMEM_ALLOC;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (CG == 2 || MC) ? 2 : 1;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    OFB_CUDA(cudaLaunchKernelEx(&cfg, corr_pyramid_kernel<T, CG, PROF, LAY, EPI, MC>, ma, mb, P));
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

// One GEMM run: queries (B, Nq, C) x targets (B, th*tw, C) -> level la of view v (th x tw per query) and, when
// has_b, its 2x2 mean, level la + 1.  layout: v's OFB_LAYOUT_*.  T: the operands' and the pyramid's 16-bit type.
template <typename T>
int run_gemm(const void* f1_km, const void* f2_km, const PyramidView& v, int layout, int la, bool has_b, int B, int C,
             int Nq, int th, int tw, float scale, int cg_mode, unsigned long long* prof, int prof_slot, cudaStream_t st) {
    // cg_mode: 1 = one CTA per tile, 2 = CTA pair sharing one 256-row accumulator tile (cta_group::2),
    //          3 = cluster of two independent cta_group::1 CTAs with the fmap2 ring multicast into both
    const bool mc = cg_mode == 3;
    const int cg = mc ? 1 : cg_mode;           // tcgen05 cta_group
    const int cl = (cg == 2 || mc) ? 2 : 1;    // CTAs per cluster / work item
    GemmParams<T> P = {};
    P.B = B; P.C = C; P.kb = C / BLOCK_K; P.Nq = Nq; P.th = th; P.tw = tw;
    P.scale = scale; P.apply_scale = (scale != 1.0f) ? 1 : 0;
    // chunk shape follows the output layout (a chunk must be whole 64/128-byte runs of it); tile shape =
    // the arrangement of 4 chunks that covers the image with the fewest tiles (ties: the widest)
    const bool blk = v.blocked;
    P.CW = blk ? 16 : 32; P.CR = blk ? 4 : 2;
    long long best = -1;
    for (int xb = 1; xb <= 4; xb *= 2) {
        const int yq = 4 / xb;
        const long long tiles = (long long)((tw + P.CW * xb - 1) / (P.CW * xb)) * ((th + P.CR * yq - 1) / (P.CR * yq));
        // measured (C3, C4, C5; profiles/): rows layout is fastest with the widest tile, blocked with 2 x 2 chunks
        const long long cost = tiles * 100 + (blk ? (xb == 2 ? 0 : 2 * tiles) : (4 - xb));
        if (best < 0 || cost < best) { best = cost; P.XB = xb; P.YQ = yq; }
    }
    if (const char* e = getenv("OFB_K2_XB")) {           // tuning override: chunks per tile row (1, 2 or 4)
        const int xb = atoi(e);
        if (xb == 1 || xb == 2 || xb == 4) { P.XB = xb; P.YQ = 4 / xb; }
    }
    const int TW = P.CW * P.XB, TH = P.CR * P.YQ;
    P.ntx = (tw + TW - 1) / TW; P.nty = (th + TH - 1) / TH; P.ntiles = P.ntx * P.nty;
    if (cl == 2) { P.nbox = P.XB >= 2 ? P.XB / 2 : 1; P.box_rows = P.XB == 1 ? TH / 2 : TH; }
    else { P.nbox = P.XB; P.box_rows = TH; }
    P.mblk = (Nq + BLOCK_M * cl - 1) / (BLOCK_M * cl);
    const int workers = ofb_num_sms() / cl;
    // split the target tiles of one (batch, query block) into chunks so the last wave is not mostly idle:
    // pick the chunk count (<= 8) that minimises ceil(items / workers) * tiles_per_item
    int best_chunks = 1;
    long long best_cost = -1;
    for (int nc = 1; nc <= 8 && nc <= P.ntiles; ++nc) {
        const int tpi = (P.ntiles + nc - 1) / nc;
        const int real_nc = (P.ntiles + tpi - 1) / tpi;
        const long long items = (long long)B * P.mblk * real_nc;
        const long long waves = (items + workers - 1) / workers;
        const long long cost = waves * (tpi + 1);   // +1: resident-A reload per item
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_chunks = real_nc; }
    }
    P.tiles_per_item = (P.ntiles + best_chunks - 1) / best_chunks;
    P.n_chunks = (P.ntiles + P.tiles_per_item - 1) / P.tiles_per_item;
    const long long n_items = (long long)B * P.mblk * P.n_chunks;
    if (n_items > 0x7fffffffLL) return OFB_EUNSUPPORTED;
    P.n_items = (int)n_items;
    P.la = level_out<T>(v, la);
    P.has_b = has_b ? 1 : 0;
    if (has_b) P.lb = level_out<T>(v, la + 1);
    P.prof = prof ? prof + (size_t)prof_slot * PROF_SLOT : nullptr;
    P.dbg = 0;
    if (prof) {
        const char* e = getenv("OFB_K2_DBG");
        if (e) P.dbg = atoi(e);
    }

    CUtensorMap ma, mb;
    {
        const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)Nq, (cuuint64_t)B};
        const cuuint64_t str[2] = {(cuuint64_t)C * 2, (cuuint64_t)Nq * C * 2};
        const cuuint32_t box[3] = {BLOCK_K, BLOCK_M, 1};
        if (!encode_tiled(&ma, F16Format<T>::tma, 3, f1_km, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
            return OFB_EDRIVER;
    }
    {
        const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)tw, (cuuint64_t)th, (cuuint64_t)B};
        const cuuint64_t str[3] = {(cuuint64_t)C * 2, (cuuint64_t)tw * C * 2, (cuuint64_t)th * tw * C * 2};
        const cuuint32_t box[4] = {BLOCK_K, (cuuint32_t)P.CW, (cuuint32_t)P.box_rows, 1};
        if (!encode_tiled(&mb, F16Format<T>::tma, 4, f2_km, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
            return OFB_EDRIVER;
    }
    int grid = workers * cl;
    if ((long long)grid > n_items * cl) grid = (int)(n_items * cl);
    if constexpr (std::is_same<T, __half>::value) {
        // fp16 is built with the direct epilogue only and has no diagnostics variant: OFB_K2_EPI is ignored here
        if (prof) return OFB_EUNSUPPORTED;
        if (mc) return layout == OFB_LAYOUT_QMINOR8X4 ? launch_gemm<T, 1, false, 2, 0, true>(ma, mb, P, grid, st)
                                                      : OFB_EUNSUPPORTED;
#define OFB_GEMM_CASE_F16(CGV, LAYV) \
        if (cg == CGV && layout == LAYV) return launch_gemm<T, CGV, false, LAYV, EPI_DIRECT, false>(ma, mb, P, grid, st);
        OFB_GEMM_CASE_F16(1, 0) OFB_GEMM_CASE_F16(1, 1) OFB_GEMM_CASE_F16(1, 2)
        OFB_GEMM_CASE_F16(2, 0) OFB_GEMM_CASE_F16(2, 1) OFB_GEMM_CASE_F16(2, 2)
#undef OFB_GEMM_CASE_F16
        return OFB_EINVAL;
    } else {
        // epilogue store mode of the query-minor layout (OFB_K2_EPI=direct|bulk overrides; other layouts stage through smem)
        int epi = EPI_DIRECT;
        if (const char* e = getenv("OFB_K2_EPI")) epi = (e[0] == 'd' || e[0] == '0') ? EPI_DIRECT : (e[0] == 'p' || e[0] == '2') ? EPI_PIPE : EPI_BULK;
        if (layout != OFB_LAYOUT_QMINOR8X4) epi = EPI_DIRECT;
#define OFB_GEMM_CASE(CGV, PROFV, LAYV, EPIV) \
        if (cg == CGV && !mc && (prof != nullptr) == PROFV && layout == LAYV && epi == EPIV) \
            return launch_gemm<T, CGV, PROFV, LAYV, EPIV, false>(ma, mb, P, grid, st);
        OFB_GEMM_CASE(1, false, 0, 0) OFB_GEMM_CASE(1, false, 1, 0) OFB_GEMM_CASE(1, false, 2, 0) OFB_GEMM_CASE(1, false, 2, 1)
        OFB_GEMM_CASE(2, false, 0, 0) OFB_GEMM_CASE(2, false, 1, 0) OFB_GEMM_CASE(2, false, 2, 0) OFB_GEMM_CASE(2, false, 2, 1)
        OFB_GEMM_CASE(1, true, 0, 0) OFB_GEMM_CASE(1, true, 1, 0) OFB_GEMM_CASE(1, true, 2, 0) OFB_GEMM_CASE(1, true, 2, 1)
        OFB_GEMM_CASE(2, true, 0, 0) OFB_GEMM_CASE(2, true, 1, 0) OFB_GEMM_CASE(2, true, 2, 0) OFB_GEMM_CASE(2, true, 2, 1)
        OFB_GEMM_CASE(1, false, 2, 2) OFB_GEMM_CASE(2, false, 2, 2) OFB_GEMM_CASE(1, true, 2, 2) OFB_GEMM_CASE(2, true, 2, 2)
        // multicast clusters: the product layout (query-minor) only
        if (mc && layout == OFB_LAYOUT_QMINOR8X4) {
            if (!prof && epi == EPI_DIRECT) return launch_gemm<T, 1, false, 2, 0, true>(ma, mb, P, grid, st);
            if (!prof && epi == EPI_BULK) return launch_gemm<T, 1, false, 2, 1, true>(ma, mb, P, grid, st);
            if (prof && epi == EPI_DIRECT) return launch_gemm<T, 1, true, 2, 0, true>(ma, mb, P, grid, st);
            if (prof && epi == EPI_BULK) return launch_gemm<T, 1, true, 2, 1, true>(ma, mb, P, grid, st);
            if (!prof && epi == EPI_PIPE) return launch_gemm<T, 1, false, 2, 2, true>(ma, mb, P, grid, st);
            if (prof && epi == EPI_PIPE) return launch_gemm<T, 1, true, 2, 2, true>(ma, mb, P, grid, st);
        }
        if (mc) return OFB_EUNSUPPORTED;
#undef OFB_GEMM_CASE
        return OFB_EINVAL;
    }
}

// dtype: the 16-bit type of the operands and of the pyramid, OFB_DTYPE_BF16 or OFB_DTYPE_F16
int corr_pyramid_impl(int dtype, const void* f1_km, const void* f2_km, const void* f2q_km, const ofb_pyramid* pyr, int B,
                      int C, int h, int w, float scale, int cta_group, unsigned long long* prof, void* stream) {
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!f1_km || !f2_km || !pyr || B < 0 || C <= 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (cta_group < 0 || cta_group > 3) return OFB_EINVAL;
    PyramidView v;
    if (const int rc = check_pyramid(pyr, (long long)B * h * w, v)) return rc;
    if (v.dtype != dtype) return OFB_EUNSUPPORTED;                     // fp32 pyramids: ofb_corr_pyramid_simt_f32
    if (C % BLOCK_K != 0 || C > MAX_KB * BLOCK_K) return OFB_EUNSUPPORTED;
    if (v.levels > 2 && !f2q_km) return OFB_EINVAL;                    // levels 2, 3 come from the 4x4-averaged fmap2
    const uintptr_t al = reinterpret_cast<uintptr_t>(f1_km) | reinterpret_cast<uintptr_t>(f2_km) |
                         reinterpret_cast<uintptr_t>(f2q_km);
    if (al & 15) return OFB_EALIGN;
    for (int l = 0; l < v.levels; ++l)      // level l of the (h, w) feature maps: (h >> l) x (w >> l)
        if (v.lh[l] != (h >> l) || v.lw[l] != (w >> l)) return OFB_EINVAL;
    const bool qminor = pyr->layout == OFB_LAYOUT_QMINOR8X4;
    for (int l = 0; l < v.levels; ++l) {
        // 16-byte store pieces: rows and query slices start on 8-element boundaries; query-minor: 32-byte sector stores
        if ((v.pitch[l] & 7) || (v.q_stride[l] & 7) || (reinterpret_cast<uintptr_t>(v.base[l]) & (qminor ? 31 : 15)))
            return OFB_EALIGN;
        const int rows = v.blocked ? ((v.lh[l] + 3) & ~3) : v.lh[l];
        if (!qminor && v.q_stride[l] < (long long)v.pitch[l] * rows) return OFB_EINVAL;
    }
    // auto (round-2 measurements, profiles/r02_k2_*.jsonl): the builder runs into the 1 kW power cap, so what pays is
    // energy per tile.  Clusters of two independent cta_group::1 CTAs with the fmap2 ring multicast into both (mode 3)
    // halve the L2 -> SM operand traffic and are 3-5 % faster than one CTA per tile at every BASELINE shape in sustained
    // runs; the CTA pair (cta_group::2) is slower (its MMAs run below the single-CTA rate and the pair's epilogues are
    // coupled through one accumulator barrier).  Mode 3 is built for the product layout only.
    int cg = cta_group;
    if (cg == 0) cg = (qminor && h * w > BLOCK_M) ? 3 : 1;
    if (cg == 3 && !qminor) return OFB_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const auto run = dtype == OFB_DTYPE_F16 ? run_gemm<__half> : run_gemm<__nv_bfloat16>;
    const int rc = run(f1_km, f2_km, v, pyr->layout, 0, v.levels > 1, B, C, h * w, h, w, scale, cg, prof, 0, st);
    if (rc != OFB_OK || v.levels <= 2) return rc;
    return run(f1_km, f2q_km, v, pyr->layout, 2, v.levels > 3, B, C, h * w, h >> 2, w >> 2, scale, cg, prof, 1, st);
}

}  // namespace

OFB_API int ofb_corr_pyramid_bf16(const void* f1_km, const void* f2_km, const void* f2q_km, const ofb_pyramid* pyr, int B,
                                  int C, int h, int w, float scale, int cta_group, void* stream) {
    return corr_pyramid_impl(OFB_DTYPE_BF16, f1_km, f2_km, f2q_km, pyr, B, C, h, w, scale, cta_group, nullptr, stream);
}

OFB_API int ofb_corr_pyramid_f16(const void* f1_km, const void* f2_km, const void* f2q_km, const ofb_pyramid* pyr, int B,
                                 int C, int h, int w, float scale, int cta_group, void* stream) {
    return corr_pyramid_impl(OFB_DTYPE_F16, f1_km, f2_km, f2q_km, pyr, B, C, h, w, scale, cta_group, nullptr, stream);
}

OFB_API int ofb_corr_pyramid_bf16_profile(const void* f1_km, const void* f2_km, const void* f2q_km, const ofb_pyramid* pyr,
                                          int B, int C, int h, int w, float scale, int cta_group, uint64_t* prof_dev,
                                          void* stream) {
    if (!prof_dev) return OFB_EINVAL;
    return corr_pyramid_impl(OFB_DTYPE_BF16, f1_km, f2_km, f2q_km, pyr, B, C, h, w, scale, cta_group,
                             reinterpret_cast<unsigned long long*>(prof_dev), stream);
}
