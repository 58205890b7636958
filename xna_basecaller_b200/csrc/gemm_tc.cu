// tcgen05 + TMA GEMM for sm_100a with fused epilogues:  D(M,N) = A(M,K) . B(N,K)^T, 16-bit K-major operands,
// fp32 accumulation in tensor memory.  One 128x128 output tile per CTA, 64-wide K blocks through a TMA ->
// mbarrier -> tcgen05.mma ring, two CTAs per SM so that one CTA's epilogue overlaps the other's main loop.
//
// Warp roles (256 threads): warp 0 = TMA producer (one elected lane), warp 1 = MMA issuer (one elected lane),
// warp 2 = TMEM allocator, warps 4..7 = epilogue (warp q reads TMEM lanes 32q..32q+31 = tile rows).
//
// Epilogues
//   EPI_F32       plain fp32 store, or fp32 atomic adds of split-K slices (weight gradients)
//   EPI_BF16OUT   plain bf16 store (gradients flowing to the layer below)
//   EPI_CONV3_BWD recomputed conv3 pre-activation -> dy * swish'(pre), bf16 in im2col row order
// The forward forms of conv3, the LSTM input projection, the CRF head and a one-launch-per-step LSTM were measured
// against the dedicated kernels and removed (DESIGN §4.3).
#include "xb_common.cuh"
#include "xb_ptx.cuh"
#include "xb_gemm.cuh"

using namespace xbptx;

namespace {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int TILE_A_BYTES = BM * BK * 2, TILE_B_BYTES = BN * BK * 2;
constexpr int STAGE_BYTES = TILE_A_BYTES + TILE_B_BYTES;
// Pipeline depth.  Three stages (96 KB) leave room for two CTAs per SM, whose epilogues and main loops overlap.
constexpr int STAGES = 3;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;

template <bool BF16, int EPI>
__global__ void __launch_bounds__(256, 2)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES);
    uint64_t *empty = full + STAGES;
    uint64_t *tmem_full = empty + STAGES;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    // K need not be a multiple of 64: the tensor maps are built over exactly K columns and TMA zero-fills the rest
    // split-K (EPI_F32 only, gridDim.z slices): slice z covers K blocks [kb0, kb0 + kblocks) and adds its partial tile to the
    // zeroed output -- for the weight-gradient contractions whose output has fewer tiles than the GPU has SMs
    const int kb_all = (p.K + BK - 1) / BK;
    const int kb_per = (kb_all + gridDim.z - 1) / gridDim.z;
    const int kb0 = blockIdx.z * kb_per;
    const int kblocks = max(0, min(kb_all, kb0 + kb_per) - kb0);

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_holder, BN);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    if (warp == 0) {
        if (elect_one()) {
            for (int kb = 0; kb < kblocks; kb++) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                mbar_expect_tx(&full[s], STAGE_BYTES);
                uint8_t *sa = smem + s * STAGE_BYTES;
                tma_load_2d(sa, &tmA, &full[s], (kb0 + kb) * BK, m0);
                tma_load_2d(sa + TILE_A_BYTES, &tmB, &full[s], (kb0 + kb) * BK, n0);
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = umma_idesc_f16(BF16 ? 1u : 0u, BM, BN);
        for (int kb = 0; kb < kblocks; kb++) {
            const int s = kb % STAGES;
            const uint32_t ph = (kb / STAGES) & 1;
            mbar_wait(&full[s], ph);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a_addr = smem_u32(smem + s * STAGE_BYTES);
                const uint32_t b_addr = a_addr + TILE_A_BYTES;
#pragma unroll
                for (int k = 0; k < BK / 16; k++) {
                    mma_f16_ss(tmem_base, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc,
                               (kb | k) != 0);
                }
                mma_commit(&empty[s]);
                if (kb == kblocks - 1) mma_commit(tmem_full);
            }
            __syncwarp();
        }
    }
    // Epilogue: warps 4..7; warp w reads TMEM lanes 32*(w%4)..+31 (= tile rows).
    __syncwarp();
    if (warp >= 4) {
        const int q = warp & 3;
        const int r = q * 32 + lane;             // tile row == TMEM lane
        const int m = m0 + r;
        const bool row_ok = m < p.M;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        if (kblocks > 0) {
            mbar_wait(tmem_full, 0);
            tc_fence_after();
        }
        if constexpr (EPI == EPI_BF16OUT) {
            // plain bf16 store of the accumulator (gradients flowing to the layer below)
#pragma unroll 1
            for (int cb = 0; cb < BN; cb += 32) {
                uint32_t acc[32];
                tmem_ld_32x32b_x32(taddr + cb, acc);
                tmem_ld_wait();
                const int nb = n0 + cb;
                if (row_ok) {
                    __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(p.out) + (size_t)m * p.ldo + nb;
                    if (nb + 32 <= p.N && (p.ldo & 7) == 0) {
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 raw;
                            __nv_bfloat162 *b2 = reinterpret_cast<__nv_bfloat162 *>(&raw);
#pragma unroll
                            for (int e = 0; e < 4; e++)
                                b2[e] = __floats2bfloat162_rn(__uint_as_float(acc[j + 2 * e]), __uint_as_float(acc[j + 2 * e + 1]));
                            *reinterpret_cast<uint4 *>(o + j) = raw;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (nb + j < p.N) o[j] = __float2bfloat16_rn(__uint_as_float(acc[j]));
                    }
                }
            }
        } else if constexpr (EPI == EPI_CONV3_BWD) {
            // conv3's pre-activation is recomputed (im2col rows x W3^T + b3) instead of stored; with the incoming gradient
            // dy (T, NB, 768) bf16 in time-major order this writes d pre = dy * swish'(pre) in im2col ROW order (chunk, t)
#pragma unroll 1
            for (int cb = 0; cb < BN; cb += 32) {
                uint32_t acc[32];
                tmem_ld_32x32b_x32(taddr + cb, acc);
                tmem_ld_wait();
                const int nb = n0 + cb;
                if (row_ok) {
                    const int b = m / p.T, t = m - b * p.T;
                    const __nv_bfloat16 *dyp = reinterpret_cast<const __nv_bfloat16 *>(p.dy) + ((size_t)t * p.NB + b) * XB_FEATURES + nb;
                    __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(p.out) + (size_t)m * p.ldo + nb;
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        const float pre = __uint_as_float(acc[j]) + __ldg(p.bias + nb + j);
                        const float sg = 1.0f / (1.0f + __expf(-pre));
                        o[j] = __float2bfloat16_rn(__bfloat162float(dyp[j]) * (sg * (1.0f + pre * (1.0f - sg))));
                    }
                }
            }
        } else if constexpr (EPI == EPI_F32) {
#pragma unroll 1
            for (int cb = 0; cb < (kblocks > 0 ? BN : 0); cb += 32) {       // an empty K slice contributes nothing
                uint32_t acc[32];
                tmem_ld_32x32b_x32(taddr + cb, acc);
                tmem_ld_wait();
                const int nb = n0 + cb;
                if (row_ok) {
                    float *o = reinterpret_cast<float *>(p.out) + (size_t)m * p.ldo + nb;
                    if (gridDim.z > 1) {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (nb + j < p.N) atomicAdd(o + j, __uint_as_float(acc[j]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (nb + j < p.N) o[j] = __uint_as_float(acc[j]);
                    }
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, BN);
    }
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

int xb_make_tmap_nd(xb_handle *h, CUtensorMap *out, const void *base, int rank, int elem_bytes, const uint64_t *dims,
                    const uint64_t *strides_bytes, const uint32_t *box, CUtensorMapSwizzle swizzle) {
    if (!h->encode_tiled) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
            return xb_fail(h, XB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
        h->encode_tiled = fn;
    }
    if (rank < 2 || rank > 5 || (elem_bytes != 2 && elem_bytes != 4)) return xb_fail(h, XB_ERR_ARG, "tensor map rank %d / element size %d", rank, elem_bytes);
    cuuint64_t d[5], st[4];
    cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; i++) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; i++) st[i] = strides_bytes[i];
    CUresult r = reinterpret_cast<encode_tiled_fn>(h->encode_tiled)(
        out, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 /* 16-bit payload; the element type only matters for OOB fill */
                             : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank,
        const_cast<void *>(base), d, st, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return xb_fail(h, XB_ERR_CUDA, "cuTensorMapEncodeTiled (rank %d) failed with CUresult %d", rank, (int)r);
    return XB_OK;
}

int xb_make_tmap_2d(xb_handle *h, CUtensorMap *out, const void *base, uint64_t rows, uint64_t K, uint64_t ld) {
    const uint64_t dims[2] = {K, rows}, strides[1] = {ld * 2};
    const uint32_t box[2] = {BK, BM};
    return xb_make_tmap_nd(h, out, base, 2, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <bool BF16, int EPI>
static int launch_one(xb_handle *h, const CUtensorMap &tmA, const CUtensorMap &tmB, const GemmParams &p, cudaStream_t s) {
    auto k = gemm_tc_kernel<BF16, EPI>;
    if (int rc = xb_smem_attr(h, k, SMEM_BYTES)) return rc;
    dim3 grid((p.N + BN - 1) / BN, (p.M + BM - 1) / BM, (EPI == EPI_F32 && p.split_k > 1) ? p.split_k : 1);
    k<<<grid, 256, SMEM_BYTES, s>>>(tmA, tmB, p);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

int xb_gemm_launch(xb_handle *h, int epi, const CUtensorMap &tmA, const CUtensorMap &tmB, const GemmParams &p,
                   cudaStream_t s, bool bf16_operands) {
    if (p.K <= 0) return xb_fail(h, XB_ERR_ARG, "GEMM K=%d", p.K);
    if (bf16_operands) {      // the training backward: gradients travel as bf16 (range), accumulated in fp32
        switch (epi) {
            case EPI_F32: return launch_one<true, EPI_F32>(h, tmA, tmB, p, s);
            case EPI_BF16OUT: return launch_one<true, EPI_BF16OUT>(h, tmA, tmB, p, s);
        }
        return xb_fail(h, XB_ERR_ARG, "no bf16 GEMM with epilogue %d", epi);
    }
    switch (epi) {      // fp16 operands in both weight modes (xb_api.cu repack)
        case EPI_F32: return launch_one<false, EPI_F32>(h, tmA, tmB, p, s);
        case EPI_CONV3_BWD: return launch_one<false, EPI_CONV3_BWD>(h, tmA, tmB, p, s);
    }
    return xb_fail(h, XB_ERR_ARG, "unknown epilogue %d", epi);
}
