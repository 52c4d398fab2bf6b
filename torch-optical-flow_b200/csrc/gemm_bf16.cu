// gemm_bf16.cu -- tcgen05 GEMMs for the backward of the correlation block, and the cast that feeds them.
//
// With dP_l the gradient of pyramid level l (queries x targets, accumulated in fp32 by lookup_bwd.cu), autograd
// through the reference's CorrBlock (methods/raft/model/corr.py:45-54,79-87: matmul, / sqrt(C), avg_pool2d chain) is
//     d fmap1[q, :]          = sum_l  sum_t dP_l[q, t] * pool_l(fmap2)[t, :] / sqrt(C)
//     d pool_l(fmap2)[t, :]  =        sum_q dP_l[q, t] * fmap1[q, :]         / sqrt(C)
// Both are D[M x N] = A[M x K] . B[N x K]^T with N = C <= 256 and a LONG K (the other spatial axis), the opposite of
// the forward builder (short K = C, huge M x N): here both operands stream through a TMA ring, the 128 x N
// accumulator lives in TMEM for the whole K loop, and the epilogue is a small fp32 store.
//   ofb_cast_bf16        fp32 (rows x cols) -> bf16 copy (A of the first product) and bf16 transpose (A of the second),
//                        row pitches padded to 8 elements (TMA strides are multiples of 16 bytes), padding zeroed
//   ofb_gemm_nt_bf16     batched D = alpha * A . B^T (+ D), bf16 K-major operands, fp32 accumulate / output
// Warp roles as in corr_gemm.cu: warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2-5 = epilogue
// (one TMEM lane quarter each); accumulators are double-buffered so the epilogue of one tile overlaps the K loop of
// the next.  Every mbarrier wait is bounded (trap instead of hang).
#include "sm100.cuh"

namespace {

using namespace ofb;

constexpr int BM = 128, BK = 64, UK = 16;
constexpr int A_STAGE = BM * BK * 2;                 // 16 KiB
constexpr int B_STAGE_MAX = 256 * BK * 2;            // 32 KiB
constexpr int STAGES = 4;
constexpr int NT = 64 + 4 * 32;                      // TMA warp, MMA warp, 4 epilogue warps
constexpr int OFF_BAR = STAGES * (A_STAGE + B_STAGE_MAX);
constexpr int NUM_BARS = 2 * STAGES + 4;
constexpr int SMEM_ALLOC = OFF_BAR + NUM_BARS * 8 + 16 + 1024;
static_assert(SMEM_ALLOC <= 232448, "shared memory budget");

struct GemmArgs {
    float* D;
    long long ldd, strideD;
    int batch, M, N, K, mtiles, kblocks, items;
    float alpha;
    int accumulate;
};

__global__ void __launch_bounds__(NT, 1) gemm_nt_kernel(const __grid_constant__ CUtensorMap map_a,
                                                        const __grid_constant__ CUtensorMap map_b, const GemmArgs G) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;       // the 128-byte swizzle is a function of the absolute address
    uint8_t* sgen = smem_raw + (sbase - raw);
    const uint32_t bar_full = sbase + OFF_BAR, bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * STAGES, bar_tempty = bar_tfull + 16;
    const uint32_t tmem_slot = sbase + OFF_BAR + NUM_BARS * 8;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(sgen + OFF_BAR + NUM_BARS * 8);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t b_stage = (uint32_t)G.N * BK * 2;
    const uint32_t off_b = STAGES * A_STAGE;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_a); prefetch_tmap(&map_b);
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(bar_tfull + 8 * s, 1); mbar_init(bar_tempty + 8 * s, 4); }
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc<1>(tmem_slot, 512);
        tmem_relinquish<1>();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int item = blockIdx.x; item < G.items; item += gridDim.x) {
                const int b = item / G.mtiles, m0 = (item - b * G.mtiles) * BM;
                for (int kb = 0; kb < G.kblocks; ++kb) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    mbar_expect_tx(bar_full + 8 * stage, (uint32_t)A_STAGE + b_stage);
                    tma_load_3d(sbase + stage * A_STAGE, &map_a, bar_full + 8 * stage, kb * BK, m0, b);
                    tma_load_3d(sbase + off_b + stage * B_STAGE_MAX, &map_b, bar_full + 8 * stage, kb * BK, 0, b);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc(BM, G.N);
            uint32_t stage = 0, phase = 0, acc = 0, tphase = 0;
            for (int item = blockIdx.x; item < G.items; item += gridDim.x) {
                mbar_wait(bar_tempty + 8 * acc, tphase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256;
                for (int kb = 0; kb < G.kblocks; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint64_t adesc = make_smem_desc(sbase + stage * A_STAGE);
                    const uint64_t bdesc = make_smem_desc(sbase + off_b + stage * B_STAGE_MAX);
#pragma unroll
                    for (int k = 0; k < BK / UK; ++k)
                        umma_bf16<1>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (uint32_t)((kb | k) != 0));
                    umma_commit<1>(bar_empty + 8 * stage);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit<1>(bar_tfull + 8 * acc);
                if (++acc == 2) { acc = 0; tphase ^= 1; }
            }
        }
        __syncwarp();
    } else {
        const int q4 = warp & 3;                          // TMEM lane quarter this warp may read (warp_id % 4)
        uint32_t acc = 0, tphase = 0;
        for (int item = blockIdx.x; item < G.items; item += gridDim.x) {
            const int b = item / G.mtiles, m0 = (item - b * G.mtiles) * BM;
            const int row = m0 + q4 * 32 + lane;
            float* drow = G.D + (long long)b * G.strideD + (long long)row * G.ldd;
            mbar_wait(bar_tfull + 8 * acc, tphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * 256;
            for (int c0 = 0; c0 < G.N; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + c0, v);
                tmem_ld_wait();
                if (row < G.M) {
#pragma unroll
                    for (int c = 0; c < 32; c += 4) {
                        float4 o = make_float4(__uint_as_float(v[c]) * G.alpha, __uint_as_float(v[c + 1]) * G.alpha,
                                               __uint_as_float(v[c + 2]) * G.alpha, __uint_as_float(v[c + 3]) * G.alpha);
                        float4* dst = reinterpret_cast<float4*>(drow + c0 + c);
                        if (G.accumulate) { const float4 p = *dst; o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w; }
                        *dst = o;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
            if (++acc == 2) { acc = 0; tphase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<1>(tmem_base, 512);
}

// fp32 (rows x cols, tight) -> bf16 copy (pitch pc) and / or bf16 transpose (pitch pr); 32 x 32 tiles through smem
__global__ void __launch_bounds__(256) cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                        __nv_bfloat16* __restrict__ dst_t, int rows, int cols, long long pc,
                                                        long long pr) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // ty 0..7
    const float* s = src + (size_t)b * rows * cols;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = r0 + ty + 8 * k, c = c0 + tx;
        const float v = (r < rows && c < cols) ? __ldg(s + (size_t)r * cols + c) : 0.0f;
        tile[ty + 8 * k][tx] = v;
        if (dst && r < rows && c < pc) dst[((size_t)b * rows + r) * pc + c] = __float2bfloat16_rn(v);
    }
    if (!dst_t) return;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + ty + 8 * k, r = r0 + tx;           // transposed: row index of dst_t = column of src
        if (c < cols && r < pr) dst_t[((size_t)b * cols + c) * pr + r] = __float2bfloat16_rn(tile[tx][ty + 8 * k]);
    }
}

bool encode_operand(CUtensorMap* m, const void* base, int K, int rows, int batch, long long ld, long long stride, int box_rows) {
    const cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)batch};
    const cuuint64_t gstr[2] = {(cuuint64_t)ld * 2, (cuuint64_t)stride * 2};
    const cuuint32_t box[3] = {BK, (cuuint32_t)box_rows, 1};
    return encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

}  // namespace

OFB_API int ofb_gemm_nt_bf16(const void* A, const void* B, float* D, int batch, int M, int N, int K, long long lda,
                             long long ldb, long long ldd, long long strideA, long long strideB, long long strideD,
                             float alpha, int accumulate, void* stream) {
    if (batch == 0 || M == 0) return OFB_OK;
    if (!A || !B || !D || batch < 0 || M < 0 || N <= 0 || K <= 0) return OFB_EINVAL;
    if (N % 32 != 0 || N > 256 || lda % 8 || ldb % 8 || strideA % 8 || strideB % 8 || ldd % 4 || strideD % 4 || lda < K || ldb < K ||
        ldd < N)
        return OFB_EUNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(D)) & 15) return OFB_EALIGN;
    CUtensorMap ma, mb;
    // batch == 1: the batch stride is unused but must still be a legal (non-zero, 16-byte multiple) stride
    const long long sa = batch > 1 ? strideA : (long long)M * lda, sb = batch > 1 ? strideB : (long long)N * ldb;
    if (!encode_operand(&ma, A, K, M, batch, lda, sa, BM) || !encode_operand(&mb, B, K, N, batch, ldb, sb, N)) return OFB_EDRIVER;
    GemmArgs G;
    G.D = D; G.ldd = ldd; G.strideD = strideD;
    G.batch = batch; G.M = M; G.N = N; G.K = K;
    G.mtiles = (M + BM - 1) / BM;
    G.kblocks = (K + BK - 1) / BK;
    const long long items = (long long)batch * G.mtiles;
    if (items > 0x7fffffffLL) return OFB_EUNSUPPORTED;
    G.items = (int)items;
    G.alpha = alpha; G.accumulate = accumulate;
    OFB_CUDA(ofb_smem_once<gemm_nt_kernel>(SMEM_ALLOC));
    const int grid = (int)(items < ofb_num_sms() ? items : ofb_num_sms());
    gemm_nt_kernel<<<grid, NT, SMEM_ALLOC, (cudaStream_t)stream>>>(ma, mb, G);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_cast_bf16(const float* src, void* dst_or_null, void* dst_t_or_null, int batch, int rows, int cols,
                          long long pitch_dst, long long pitch_dst_t, void* stream) {
    if (batch == 0 || rows == 0 || cols == 0) return OFB_OK;
    if (!src || (!dst_or_null && !dst_t_or_null) || batch < 0 || rows < 0 || cols < 0) return OFB_EINVAL;
    if ((dst_or_null && pitch_dst < cols) || (dst_t_or_null && pitch_dst_t < rows)) return OFB_EINVAL;
    // the padding is written from the same tiles: it may extend at most to the next multiple of 32
    const long long cmax = ((long long)cols + 31) / 32 * 32, rmax = ((long long)rows + 31) / 32 * 32;
    if ((dst_or_null && pitch_dst > cmax) || (dst_t_or_null && pitch_dst_t > rmax) || batch > 65535) return OFB_EUNSUPPORTED;
    const dim3 grid((cols + 31) / 32, (rows + 31) / 32, batch);
    if (grid.y > 65535) return OFB_EUNSUPPORTED;
    cast_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, static_cast<__nv_bfloat16*>(dst_or_null),
                                                            static_cast<__nv_bfloat16*>(dst_t_or_null), rows, cols, pitch_dst,
                                                            pitch_dst_t);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
