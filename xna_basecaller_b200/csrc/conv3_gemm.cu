// Third Convolution of the stem (bonito/nn.py:57-68: Conv1d(16, 768, 19, stride 5, padding 9) + swish, followed by
// nn.Permute([2,0,1]), nn.py:156-167) as a WEIGHT-STATIONARY persistent tcgen05 GEMM over the im2col rows of conv_stem.cu:
//
//   out[t, b, :] = swish( col[(b, t), 0:320] . W3^T + b3 )          M = N*T rows, K = 320 (16 channels x 19 taps + pad), 768 columns
//
// Why not the generic tile kernel (a conv3 epilogue of gemm_tc.cu was measured at 0.48 ms per 512-chunk batch and removed).
// With K = 320 a 128 x 128 output tile moves 80 KB of im2col rows and 80 KB of weights for 1280 MMA cycles: 2600 cycles of
// L2 ingest at ~62 B/clk per SM, and the im2col matrix is read six times (once per column tile).  Here each CTA keeps a 192-column slice of W3 (120 KB)
// in shared memory for its whole life and streams only im2col row tiles (80 KB per 128 x 192 outputs = 1920 MMA cycles):
// the kernel is bound by the tensor pipe and its epilogue instead of by ingest.
//
// Grid: 4 column groups x 37 workers = 148 CTAs, one per SM; worker w of a group takes row tiles w, w + 37, ...
// Two 192-column fp32 accumulators in tensor memory: the epilogue of row tile i (one of two sets of four warps, taking
// alternate tiles) overlaps the MMAs of tile i + 1.  The epilogue adds the bias, applies swish with one MUFU per element,
// stages 32 x 64 fp16 blocks with the 128-byte swizzle and lets TMA write them into the (T, N, 768) output -- the
// (chunk, t) -> (t, chunk) row permutation is the tensor map's stride.  A block that crosses from chunk b into chunk b + 1
// (only when T is not a multiple of 32; never at T = 800) is copied row by row instead.
//
// Warp roles (384 threads): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4..7 / 8..11 epilogue
// sets 0 / 1 (warp % 4 = TMEM lane quarter).
#include "xb_common.cuh"
#include "xb_ptx.cuh"
#include "xb_gemm.cuh"

using namespace xbptx;

namespace {

constexpr int BM = 128, BN = 192, BK = 64;
constexpr int KBLK = XB_CONV3_K / BK;                       // 5
constexpr int GROUPS = XB_FEATURES / BN;                    // 4
constexpr int A_BYTES = BM * BK * 2, B_KB_BYTES = BN * BK * 2;
constexpr int STAGES = 4;
constexpr int STG_BYTES = 32 * 128;                         // one warp's staged [32 rows x 64 fp16] block
constexpr int OFF_A = KBLK * B_KB_BYTES;                    // 120 KB of resident weights, then the row-tile ring
constexpr int OFF_STG = OFF_A + STAGES * A_BYTES;
constexpr int OFF_BIAS = OFF_STG + 8 * STG_BYTES;
constexpr int OFF_BAR = OFF_BIAS + BN * 4;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024 /*align slack*/;
constexpr int THREADS = 384;
static_assert(XB_CONV3_K % BK == 0 && XB_FEATURES % BN == 0, "tile plan");
static_assert(OFF_A % 1024 == 0 && OFF_STG % 1024 == 0 && SMEM_BYTES <= 232448, "shared memory plan");

struct Conv3Params {
    int M, T, NB;            // im2col rows (= NB * T), steps per chunk, chunks
    const float *bias;       // (768)
    const void *col;         // the im2col rows (for the L2 prefetch; the loads go through the tensor map)
    uint16_t *out;           // (T, NB, 768) fp16 (the TMA stores go through the tensor map; rows of blocks that cross a chunk edge do not)
};

__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap *m, uint32_t src_smem, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(m), "r"(src_smem), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

__global__ void __launch_bounds__(THREADS, 1)
conv3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmO, const Conv3Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    float *sbias = reinterpret_cast<float *>(smem + OFF_BIAS);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
    uint64_t *empty = full + STAGES;
    uint64_t *acc_full = empty + STAGES;       // [2]
    uint64_t *acc_empty = acc_full + 2;        // [2]
    uint64_t *w_full = acc_empty + 2;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(w_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int group = blockIdx.x % GROUPS, worker = blockIdx.x / GROUPS, workers = gridDim.x / GROUPS;
    const int n0 = group * BN;
    const int ntiles = (p.M + BM - 1) / BM;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
        prefetch_tmap(&tmO);
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 4);
        }
        mbar_init(w_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_holder, 512);
        tmem_relinquish();
    }
    for (int i = threadIdx.x; i < BN; i += THREADS) sbias[i] = p.bias[n0 + i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    if (warp == 0) {
        if (elect_one()) {
            mbar_expect_tx(w_full, KBLK * B_KB_BYTES);
            for (int kb = 0; kb < KBLK; kb++) tma_load_2d(smem + kb * B_KB_BYTES, &tmB, w_full, kb * BK, n0);
            uint32_t it = 0;
            for (int tile = worker; tile < ntiles; tile += workers) {
                // The im2col matrix (262 MB at N = 512) does not stay in L2, and four stages of 16 KB in flight cannot cover an
                // HBM round trip at the rate the tensor pipe drains them: pull the row tile after the next one (128 rows x 640 B,
                // contiguous) into L2 now, so that the ring only ever waits for L2.  One group does it for all four.
                const int ahead = tile + 2 * workers;
                if (group == 0 && ahead < ntiles) {
                    const int rows = min(BM, p.M - ahead * BM);
                    const char *src = reinterpret_cast<const char *>(p.col) + (size_t)ahead * BM * (XB_CONV3_K * 2);
                    const uint32_t bytes = (uint32_t)rows * (XB_CONV3_K * 2);
                    for (uint32_t off = 0; off < bytes; off += 16384) prefetch_l2_bulk(src + off, min(16384u, bytes - off));
                }
                for (int kb = 0; kb < KBLK; kb++, it++) {
                    const int s = it % STAGES;
                    mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                    mbar_expect_tx(&full[s], A_BYTES);
                    tma_load_2d(smem + OFF_A + s * A_BYTES, &tmA, &full[s], kb * BK, tile * BM);
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = umma_idesc_f16(0u, BM, BN);
        mbar_wait(w_full, 0);
        uint32_t it = 0, ti = 0;
        for (int tile = worker; tile < ntiles; tile += workers, ti++) {
            const int buf = ti & 1;
            mbar_wait(&acc_empty[buf], ((ti >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d = tmem_base + buf * BN;
            for (int kb = 0; kb < KBLK; kb++, it++) {
                const int s = it % STAGES;
                mbar_wait(&full[s], (it / STAGES) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_addr = smem_u32(smem + OFF_A + s * A_BYTES);
                    const uint32_t b_addr = smem_u32(smem + kb * B_KB_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / 16; k++)
                        mma_f16_ss(d, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc, (kb | k) != 0);
                    mma_commit(&empty[s]);
                    if (kb == KBLK - 1) mma_commit(&acc_full[buf]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= 4) {
        const int set = (warp - 4) >> 2, q = warp & 3;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const uint32_t stg = smem_u32(smem + OFF_STG + (set * 4 + q) * STG_BYTES);
        const uint32_t row_s = stg + lane * 128;
        uint32_t ti = 0;
        for (int tile = worker; tile < ntiles; tile += workers, ti++) {
            if ((int)(ti & 1) != set) continue;                  // the other set's tile
            const int buf = ti & 1;
            mbar_wait(&acc_full[buf], (ti >> 1) & 1);
            tc_fence_after();
            // first row of this warp's block and where it lives in the (T, NB, 768) output
            const int m_w = tile * BM + q * 32;
            const int b_w = m_w / p.T, t_w = m_w - b_w * p.T;
#pragma unroll 1
            for (int cb = 0; cb < BN; cb += 64) {
                uint32_t a0[32], a1[32];
                tmem_ld_32x32b_x32(lane_base + buf * BN + cb, a0);
                tmem_ld_32x32b_x32(lane_base + buf * BN + cb + 32, a1);
                tmem_ld_wait();
                if (cb + 64 == BN) {                             // accumulator drained: the MMAs of tile ti + 2 may overwrite it
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[buf]);
                }
                const float *bs = sbias + cb;
                uint32_t pk[32];                                 // the thread's 64 activated columns, packed fp16
#pragma unroll
                for (int e = 0; e < 32; e++) {
                    const int c = 2 * e;
                    float v0 = __uint_as_float(c < 32 ? a0[c & 31] : a1[c & 31]) + bs[c];
                    float v1 = __uint_as_float(c < 32 ? a0[(c + 1) & 31] : a1[(c + 1) & 31]) + bs[c + 1];
                    v0 = v0 * fmaf(tanh_approx(0.5f * v0), 0.5f, 0.5f);          // swish, sigmoid(x) = 0.5 tanh(0.5 x) + 0.5
                    v1 = v1 * fmaf(tanh_approx(0.5f * v1), 0.5f, 0.5f);
                    pk[e] = xb16<false>::pack(v0, v1);
                }
                if (lane == 0) bulk_wait_group_read0();          // the previous block has left the staging rows (its store ran
                __syncwarp();                                    // under the arithmetic above)
#pragma unroll
                for (int j = 0; j < 8; j++)                      // 8 columns = one 16-byte chunk of the staged row
                    sts_v4(row_s + (uint32_t)((j ^ (lane & 7)) << 4), make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]));
                if (t_w + 32 <= p.T) {                           // the whole block lies in chunk b_w: one TMA store
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (b_w < p.NB) tma_store_3d(&tmO, stg, n0 + cb, t_w, b_w);
                        bulk_commit_group();
                    }
                } else {
                    // the block crosses into the next chunk (only when T is not a multiple of 32) or past the last row: every
                    // lane copies its own row to where it lives, 8 x 16 bytes
                    __syncwarp();
                    const int m = m_w + lane;
                    if (m < p.M) {
                        const int b = m / p.T, t = m - b * p.T;
                        uint16_t *o = p.out + ((size_t)t * p.NB + b) * XB_FEATURES + n0 + cb;
#pragma unroll
                        for (int j = 0; j < 8; j++)
                            reinterpret_cast<uint4 *>(o)[j] = lds_v4(row_s + (uint32_t)((j ^ (lane & 7)) << 4));
                    }
                    __syncwarp();
                }
            }
        }
        if (lane == 0) bulk_wait_group0();
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

}  // namespace

// col: (N*T, 320) fp16 im2col rows in (chunk, t) order; w3: (768, 320) fp16; out: (T, N, 768) fp16
int xb_conv3_launch(xb_handle *h, const void *col, const void *w3, const float *bias, void *out_tnc, int T, int N, cudaStream_t s) {
    const uint64_t M = (uint64_t)N * T;
    CUtensorMap tmA, tmB, tmO;
    if (int rc = xb_make_tmap_2d(h, &tmA, col, M, XB_CONV3_K, XB_CONV3_K)) return rc;
    {
        const uint64_t dims[2] = {XB_CONV3_K, XB_FEATURES}, st[1] = {XB_CONV3_K * 2};
        const uint32_t box[2] = {BK, BN};
        if (int rc = xb_make_tmap_nd(h, &tmB, w3, 2, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    {
        const uint64_t dims[3] = {XB_FEATURES, (uint64_t)T, (uint64_t)N};
        const uint64_t st[2] = {(uint64_t)N * XB_FEATURES * 2, XB_FEATURES * 2};
        const uint32_t box[3] = {64, 32, 1};
        if (int rc = xb_make_tmap_nd(h, &tmO, out_tnc, 3, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    if (int rc = xb_smem_attr(h, conv3_kernel, SMEM_BYTES)) return rc;
    Conv3Params p;
    p.M = (int)M; p.T = T; p.NB = N; p.bias = bias; p.col = col; p.out = reinterpret_cast<uint16_t *>(out_tnc);
    const int ntiles = (int)((M + BM - 1) / BM);
    int workers = (h->num_sms > 0 ? h->num_sms : 148) / GROUPS;       // one CTA per SM
    if (workers > ntiles) workers = ntiles;
    conv3_kernel<<<GROUPS * workers, THREADS, SMEM_BYTES, s>>>(tmA, tmB, tmO, p);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
