// Weight gradients of one LSTM layer in one launch (the backward of bonito/nn.py:189-193's torch.nn.LSTM):
//
//   dW_ih (3072, 768) = DZ^T X            K = T*N            (X = the layer's input,  transposed copy XT (768, T*N))
//   dW_hh (3072, 768) = DZ^T H_prev       K = T*N - N        (H_prev = the layer's output one step earlier, YT (768, T*N))
//
// as ONE (3072 x 1536) product over 128 x 256 output tiles: 24 x 6 = 144 CTAs, one per SM, fp32 accumulators in 256 columns
// of tensor memory.  Both contractions are bound by what one SM can ingest from L2 (~62 B/clk): a 128 x 128 tile moves
// 32 KB per 64-deep K block for 1 M MACs, a 128 x 256 tile 48 KB for 2 M -- the two 128 x 128-tile GEMMs this replaces took
// 2 x 2.8 ms per layer.  Column tiles 0-2 are dW_ih, 3-5 dW_hh; the time shift of dW_hh is a K-coordinate offset on one
// operand (forward layers: DZ^T shifted by +N, reverse layers: Y^T shifted by +N), and the N columns that fall off the end
// are zero-filled by TMA, so both halves run the same K = T*N loop.
#include "xb_common.cuh"
#include "xb_ptx.cuh"
#include "xb_gemm.cuh"

using namespace xbptx;

namespace {

constexpr int BM = 128, BN = 256, BK = 64;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int STAGES = 4;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;

struct WgradParams {
    int K;                  // T*N
    int a_shift, b_shift;   // K-coordinate offsets of the dW_hh half (one of them is N, the other 0)
    float *out_ih, *out_hh; // (3072, 768) fp32 each
};

__global__ void __launch_bounds__(256, 1)
lstm_wgrad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmX,
                  const __grid_constant__ CUtensorMap tmY, const WgradParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES);
    uint64_t *empty = full + STAGES;
    uint64_t *tmem_full = empty + STAGES;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool hh = blockIdx.x >= XB_FEATURES / BN;                    // column tiles 3..5: the recurrent weights
    const int n0 = (hh ? blockIdx.x - XB_FEATURES / BN : blockIdx.x) * BN, m0 = blockIdx.y * BM;
    const CUtensorMap *tmB = hh ? &tmY : &tmX;
    const int a_shift = hh ? p.a_shift : 0, b_shift = hh ? p.b_shift : 0;
    const int kblocks = (p.K + BK - 1) / BK;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(tmB);
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
                mbar_wait(&empty[s], ((kb / STAGES) & 1) ^ 1);
                mbar_expect_tx(&full[s], STAGE_BYTES);
                uint8_t *sa = smem + s * STAGE_BYTES;
                tma_load_2d(sa, &tmA, &full[s], kb * BK + a_shift, m0);
                tma_load_2d(sa + A_BYTES, tmB, &full[s], kb * BK + b_shift, n0);
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = umma_idesc_f16(1u, BM, BN);
        for (int kb = 0; kb < kblocks; kb++) {
            const int s = kb % STAGES;
            mbar_wait(&full[s], (kb / STAGES) & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a_addr = smem_u32(smem + s * STAGE_BYTES);
                const uint32_t b_addr = a_addr + A_BYTES;
#pragma unroll
                for (int k = 0; k < BK / 16; k++)
                    mma_f16_ss(tmem_base, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc, (kb | k) != 0);
                mma_commit(&empty[s]);
                if (kb == kblocks - 1) mma_commit(tmem_full);
            }
            __syncwarp();
        }
    }
    __syncwarp();
    {
        // all eight warps: warp w reads TMEM lanes 32 (w % 4) .. + 31 (= tile rows), columns 128 (w / 4) .. + 127
        const int q = warp & 3, half = warp >> 2;
        const int m = m0 + q * 32 + lane;
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        float *o = (hh ? p.out_hh : p.out_ih) + (size_t)m * XB_FEATURES + n0 + half * 128;
#pragma unroll 1
        for (int cb = 0; cb < 128; cb += 32) {
            uint32_t acc[32];
            tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + half * 128 + cb, acc);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4 *>(o + cb + j) = make_float4(__uint_as_float(acc[j]), __uint_as_float(acc[j + 1]),
                                                                      __uint_as_float(acc[j + 2]), __uint_as_float(acc[j + 3]));
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, BN);
    }
}

}  // namespace

// dzT (3072, TN) bf16, xT / yT (768, TN) bf16; reverse: the layer ran t = T-1 .. 0 (its predecessor step is t + 1)
int xb_lstm_wgrad_launch(xb_handle *h, const void *dzT, const void *xT, const void *yT, int T, int N, bool reverse, float *g_wih,
                         float *g_whh, cudaStream_t s) {
    const uint64_t TN = (uint64_t)T * N;
    CUtensorMap tmA, tmX, tmY;
    const uint64_t dims_dz[2] = {TN, XB_GATES}, dims_h[2] = {TN, XB_FEATURES}, st[1] = {TN * 2};
    const uint32_t box_dz[2] = {BK, BM}, box_h[2] = {BK, BN};
    if (int rc = xb_make_tmap_nd(h, &tmA, dzT, 2, 2, dims_dz, st, box_dz, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = xb_make_tmap_nd(h, &tmX, xT, 2, 2, dims_h, st, box_h, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = xb_make_tmap_nd(h, &tmY, yT, 2, 2, dims_h, st, box_h, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = xb_smem_attr(h, lstm_wgrad_kernel, SMEM_BYTES)) return rc;
    WgradParams p;
    p.K = (int)TN;
    // forward layers: steps t = 1 .. T-1 pair dz_t with h_{t-1}:  DZ^T column k + N  x  Y^T column k
    // reverse layers: steps t = 0 .. T-2 pair dz_t with h_{t+1}:  DZ^T column k      x  Y^T column k + N
    p.a_shift = reverse ? 0 : N;
    p.b_shift = reverse ? N : 0;
    p.out_ih = g_wih;
    p.out_hh = g_whh;
    lstm_wgrad_kernel<<<dim3(2 * XB_FEATURES / BN, XB_GATES / BM), 256, SMEM_BYTES, s>>>(tmA, tmX, tmY, p);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
