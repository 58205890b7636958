// LSTM input projection G = x W_ih^T + (b_ih + b_hh) for all T*N rows at once (the hoisted half of
// torch.nn.LSTM, bonito/nn.py:189-193), as an A-STATIONARY persistent tcgen05 GEMM.
//
// Why not the generic tile kernel (gemm_tc.cu).  A B200 SM ingests ~64 B/clk from L2 while its tensor core
// retires 8192 dense 16-bit FLOP/clk.  A 128x128 output tile with K = 768 needs 2 x 196 KB of operands for 3072
// MMA cycles: 6144 cycles of ingest, so that kernel runs ingest-bound at <= 50% of the tensor peak (measured
// 37%).  Here the 128 x 768 block of x rows is loaded ONCE per M tile into TENSOR MEMORY (384 of the 512
// columns; the A operand of tcgen05.mma) and only W_ih streams through shared memory: 96 KB per 64-column
// N tile for 1536 MMA cycles -- ingest and tensor time balance, and x is read from HBM exactly once.
//
// One CTA per SM, persistent over M tiles (tile = blockIdx.x, += gridDim.x).  Per M tile: 48 N tiles of 64
// gate columns; two 64-column fp32 accumulators in the remaining 128 TMEM columns, so the epilogue of N tile i
// (TMEM -> +bias -> 16-bit -> staged rows -> 128-byte row segments of G) overlaps the MMAs of N tile i+1.
// W_ih arrives as 3-D TMA boxes of four [64 rows x 64 K] 128B-swizzled blocks (32 KB) through a 6-stage ring
// (192 KB in flight); one mbarrier wait and one commit per 16 MMAs keep the single issuing thread ahead of
// the tensor pipe (with one wait per 4 MMAs the issue loop, not the pipe, set the pace).  The x block travels through
// the same ring (six stages of two [128 rows x 64 K] blocks in front of every tile's W stages) and is copied into
// tensor memory with tcgen05.cp by the MMA thread, in issue order with its MMAs.
//
// The same kernel with the IP_SCORES epilogue is the CRF head (LinearCRFEncoder, nn.py:87-133): W_head streams instead
// of W_ih, fp32 score rows with the blank score inserted leave as coalesced segments, two epilogue warp sets.
//
// Warp roles (256 threads; 384 for IP_SCORES): warp 0 TMA producer, warp 1 MMA issuer (+ tcgen05.cp of the x block),
// warp 2 TMEM allocator, warps 4..7 (and 8..11) run the epilogues (warp % 4 = TMEM lane quarter).  The earlier x path
// (epilogue warps load the rows, transpose them through staging rows, tcgen05.st) was measured and removed (DESIGN §4.2).
#include "xb_common.cuh"
#include "xb_ptx.cuh"
#include "xb_gemm.cuh"
#include "xb_exact_math.h"

using namespace xbptx;

namespace {

constexpr int BM = 128, BNI = 64, BK = 64;
constexpr int KB = XB_FEATURES / BK;                 // 12 K blocks
constexpr int MAX_COLS = XB_GATES;                   // most output columns (rows of W) a launch handles: 48 N tiles
constexpr int KPS = 4;                               // K blocks per pipeline stage (one 3-D TMA box, 16 MMAs per wait)
constexpr int SPT = KB / KPS;                        // stages per N tile
enum { IP_GATES = 0, IP_SCORES = 1 };                // epilogue: 16-bit gates (+bias) | fp32 CRF scores (LinearCRFEncoder)
template <int EPI> struct IPCfg {
    static constexpr int STAGES = EPI == IP_GATES ? 6 : 4;
    static constexpr int SETS = EPI == IP_GATES ? 1 : 2;     // epilogue warp sets (4 warps each) taking alternate accumulators
    static constexpr int THREADS = (4 + 4 * SETS) * 32;
    static constexpr int STG_BYTES = EPI == IP_GATES ? 32 * (BNI * 2 + 16) : 32 * 81 * 4;     // per epilogue warp
    static constexpr int SMEM_BYTES = STAGES * (KPS * BNI * BK * 2) + 4 * SETS * STG_BYTES + MAX_COLS * 4 + 1024 /*align*/ + 512 /*barriers*/;
};
constexpr int KBLOCK_BYTES = BNI * BK * 2;           // 8 KB: one [64 rows x 128 B] swizzle atom column
constexpr int STAGE_BYTES = KPS * KBLOCK_BYTES;      // 32 KB
constexpr int A_COLS = XB_FEATURES / 2;              // 384 TMEM columns hold the x block
constexpr int ROW_PITCH = BNI * 2 + 16;              // staged epilogue row pitch (bytes)

struct IPParams {
    const uint16_t *x;        // (M, 768) 16-bit
    const float *bias;        // (n_valid) fp32, same column order as the rows of W
    void *out;                // IP_GATES: (M, ldo) 16-bit; IP_SCORES: (M, ldo) fp32
    int M;
    int NT;                   // N tiles of 64 columns (rows of W, zero padded to a multiple of 64)
    int n_valid, ldo;         // valid output columns before expansion; output row pitch in elements
    int n_base, expand;       // IP_SCORES: blank score inserted in front of every n_base columns
    float scale, blank;
    int exp_out;              // IP_SCORES: write E = xb_score_exp(score) (what the linear-domain decode consumes) instead of the score
};

// LinearCRFEncoder (nn.py:117-129): scale * tanh(acc + bias), with the blank score written in front of every group of
// n_base columns.
__device__ __forceinline__ float fast_tanh(float x) { return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f); }

// Output positions [seg_start, seg_start + seg_len) covered by head columns [col0, col_end).
__device__ __forceinline__ void segment(int col0, int col_end, int nbs, int expand, int &seg_start, int &seg_len) {
    seg_start = 0; seg_len = 0;
    if (col_end <= col0) return;
    if (expand) {
        seg_start = col0 + col0 / nbs + ((col0 % nbs) ? 1 : 0);
        seg_len = (col_end - 1) + (col_end - 1) / nbs + 2 - seg_start;
    } else {
        seg_start = col0;
        seg_len = col_end - col0;
    }
}

// LinearCRFEncoder expansion of one thread's 64 activated columns into its staged row (shared address sr, positions
// relative to the segment start): column jj of the tile goes to pos0 + jj + (e0 + jj) / NB, the blank score in front of
// every column that starts a group.  NB compile-time (division by a constant), explicit st.shared (through the lambda the
// compiler had lost the address space and emitted generic stores with 64-bit address arithmetic and a branch per column).
template <int NB, bool FULL>
__device__ __forceinline__ void head_stage64(const float (&v)[BNI], uint32_t sr, int e0, int pos0, int ncols, float blank) {
#pragma unroll
    for (int jj = 0; jj < BNI; jj++) {
        if (FULL || jj < ncols) {
            const unsigned u = (unsigned)(e0 + jj);
            const unsigned g = u / NB;
            const uint32_t a = sr + 4u * (uint32_t)(pos0 + jj + (int)g);
            sts_f32(a, v[jj]);
            if (u - g * NB == 0) sts_f32(a - 4u, blank);
        }
    }
}
template <bool FULL>
__device__ __forceinline__ void head_stage64_dyn(const float (&v)[BNI], uint32_t sr, int nb, int e0, int pos0, int ncols, float blank) {
    int e = e0, o = pos0;
#pragma unroll
    for (int jj = 0; jj < BNI; jj++) {
        if (FULL || jj < ncols) {
            if (e == 0) sts_f32(sr + 4u * (uint32_t)(o - 1), blank);
            sts_f32(sr + 4u * (uint32_t)o, v[jj]);
            o++;
            if (++e == nb) { e = 0; o++; }
        }
    }
}

// The x block reaches tensor memory as TMA boxes (two K blocks = one 32 KB ring stage, interleaved with the W stages by
// the producer) copied with tcgen05.cp by the MMA thread, in issue order with its MMAs -- no register / staging-row detour
// through the epilogue warps, and the next tile's x stages are already in flight while the current tile finishes
// (tools/tmem_cp_probe.cu checks the copy's layout: lane = row, column c = elements 2c, 2c+1, as the TS-mode MMA reads A).
template <int EPI>
__global__ void __launch_bounds__(IPCfg<EPI>::THREADS, 1)
inproj_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX, const IPParams p) {
    using X = xb16<false>;                    // fp16 operands in both weight modes (xb_api.cu repack)
    constexpr int STAGES = IPCfg<EPI>::STAGES, STG_BYTES = IPCfg<EPI>::STG_BYTES;
    const int NT = p.NT;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *stgbuf = smem + STAGES * STAGE_BYTES;
    float *sbias = reinterpret_cast<float *>(stgbuf + 4 * IPCfg<EPI>::SETS * STG_BYTES);
    uint64_t *full = reinterpret_cast<uint64_t *>(sbias + MAX_COLS);
    uint64_t *empty = full + STAGES;
    uint64_t *acc_full = empty + STAGES;      // [2]
    uint64_t *acc_empty = acc_full + 2;       // [2]
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(acc_empty + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int ntiles = (p.M + BM - 1) / BM;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmW);
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 4);
        }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_holder, 512);
        tmem_relinquish();
    }
    for (int i = threadIdx.x; i < NT * BNI; i += IPCfg<EPI>::THREADS) sbias[i] = i < p.n_valid ? p.bias[i] : 0.0f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer: W_ih boxes, all tiles
        if (elect_one()) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                for (int xs = 0; xs < KB / 2; xs++, it++) {                // x block: [128 rows x 64 K] x 2 K blocks per stage
                    const int s = it % STAGES;
                    mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                    mbar_expect_tx(&full[s], STAGE_BYTES);
                    tma_load_3d(smem + s * STAGE_BYTES, &tmX, &full[s], 0, tile * BM, xs * 2);
                }
                for (int nt = 0; nt < NT; nt++)
                    for (int ks = 0; ks < SPT; ks++, it++) {
                        const int s = it % STAGES;
                        mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                        mbar_expect_tx(&full[s], STAGE_BYTES);
                        tma_load_3d(smem + s * STAGE_BYTES, &tmW, &full[s], 0, nt * BNI, ks * KPS);
                    }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        constexpr uint32_t idesc = umma_idesc_f16(0u, BM, BNI);
        uint32_t it = 0, nit = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            for (int xs = 0; xs < KB / 2; xs++, it++) {
                const int s = it % STAGES;
                mbar_wait(&full[s], (it / STAGES) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t sdesc = umma_desc_sw128(smem_u32(smem + s * STAGE_BYTES));
#pragma unroll
                    for (int kk = 0; kk < 8; kk++)                 // 2 K blocks x 4 slices of K = 16: 8 tensor-memory columns each
                        tmem_cp_128x256b(tmem_base + (xs * 2) * (BK / 2) + kk * 8,
                                         sdesc + (uint64_t)(((kk >> 2) * (BM * BK * 2) + (kk & 3) * 32) >> 4));
                    mma_commit(&empty[s]);
                }
                __syncwarp();
            }
            for (int nt = 0; nt < NT; nt++, nit++) {
                const int buf = nit & 1;
                mbar_wait(&acc_empty[buf], ((nit >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d = tmem_base + A_COLS + buf * BNI;
                for (int ks = 0; ks < SPT; ks++, it++) {
                    const int s = it % STAGES;
                    mbar_wait(&full[s], (it / STAGES) & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint64_t bdesc = umma_desc_sw128(smem_u32(smem + s * STAGE_BYTES));
                        const uint32_t a0 = tmem_base + ks * KPS * (BK / 2);
#pragma unroll
                        for (int kk = 0; kk < KPS * 4; kk++) {
                            const int kc = kk >> 2, k = kk & 3;
                            mma_f16_ts(d, a0 + kk * 8, bdesc + (uint64_t)((kc * KBLOCK_BYTES + k * 32) >> 4), idesc,
                                       (ks | kk) != 0);
                        }
                        mma_commit(&empty[s]);
                        if (ks == SPT - 1) mma_commit(&acc_full[buf]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue
        // Scores variant: two sets of four warps; set s runs the epilogues of the accumulators with (N-tile counter & 1) == s,
        // so consecutive epilogues overlap (each is several times longer than the MMAs of an N tile).
        constexpr int SETS = IPCfg<EPI>::SETS;
        const int set = (warp - 4) >> 2;
        const int q = warp & 3, r = q * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        uint8_t *stg = stgbuf + (set * 4 + q) * STG_BYTES;
        const uint32_t stg_s = smem_u32(stg);          // explicit shared addressing: through the lambdas the compiler falls back to generic loads / stores
        uint32_t nit = 0;
        bool pending = false;                                  // epilogue of the previous tile's last N tile
        int pend_m0 = 0;

        auto epilogue = [&](int m0, int nt, uint32_t ni) {
            const int buf = ni & 1;
            uint32_t acc[BNI];
            {
                uint32_t a0[32], a1[32];
                tmem_ld_32x32b_x32(lane_base + A_COLS + buf * BNI, a0);
                tmem_ld_32x32b_x32(lane_base + A_COLS + buf * BNI + 32, a1);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; i++) { acc[i] = a0[i]; acc[32 + i] = a1[i]; }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);       // the MMAs of N tile ni+2 may overwrite it now
            if constexpr (EPI == IP_GATES) {
                const float *bs = sbias + nt * BNI;
    #pragma unroll
                for (int j = 0; j < BNI / 8; j++) {
                    uint32_t pk[4];
    #pragma unroll
                    for (int e = 0; e < 4; e++)
                        pk[e] = X::pack(__uint_as_float(acc[8 * j + 2 * e]) + bs[8 * j + 2 * e],
                                        __uint_as_float(acc[8 * j + 2 * e + 1]) + bs[8 * j + 2 * e + 1]);
                    sts_v4(stg_s + lane * ROW_PITCH + j * 16, make_uint4(pk[0], pk[1], pk[2], pk[3]));
                }
                __syncwarp();
                const int sub = lane >> 3, l8 = lane & 7;          // 8 lanes x 16 B = one 128-byte row segment
    #pragma unroll
                for (int rr = 0; rr < 32; rr += 4) {
                    const int mm = m0 + q * 32 + rr + sub;
                    if (mm < p.M)
                        reinterpret_cast<uint4 *>(reinterpret_cast<uint16_t *>(p.out) + (size_t)mm * p.ldo + nt * BNI)[l8] =
                            lds_v4(stg_s + (rr + sub) * ROW_PITCH + l8 * 16);
                }
            } else {
                // LinearCRFEncoder: scale * tanh(acc + bias), blank score in front of every group of n_base columns; the
                // thread's row goes to a staged row (odd pitch: conflict free), rows leave as coalesced fp32 segments
                constexpr int RS = 81;
                float *S = reinterpret_cast<float *>(stg);
                const int col0 = nt * BNI, col_end = min(col0 + BNI, p.n_valid);
                int seg_start, seg_len;
                segment(col0, col_end, p.n_base, p.expand, seg_start, seg_len);
                if (seg_len > 0) {
                    // activation first (64 independent MUFU chains), then the expansion with running positions: no
                    // compile-time variants per (n_base, group phase) here -- the issue slots are idle anyway, the instruction
                    // cache is not
                    const float *bs = sbias + col0;
                    float v[BNI];
#pragma unroll
                    for (int jj = 0; jj < BNI; jj++) v[jj] = p.scale * fast_tanh(__uint_as_float(acc[jj]) + bs[jj]);
                    // fused pipeline: hand the decode exp(score) -- the one exponential per edge its three sweeps would
                    // otherwise each compute (bit-reproducible xb_score_exp, the decode contract's own function)
                    if (p.exp_out) {
#pragma unroll
                        for (int jj = 0; jj < BNI; jj++) v[jj] = xb_score_exp(v[jj]);
                    }
                    const float blank = p.exp_out ? xb_score_exp(p.blank) : p.blank;
                    const uint32_t sr = smem_u32(S) + (uint32_t)(lane * RS * 4);
                    const int ncols = col_end - col0;
                    if (p.expand) {
                        const int nb = p.n_base, c = col0 / nb, e0 = col0 - c * nb;
                        const int pos0 = col0 + c + 1 - seg_start;         // staged position of column col0
                        if (ncols == BNI) {
                            if (nb == 5) head_stage64<5, true>(v, sr, e0, pos0, ncols, blank);
                            else if (nb == 4) head_stage64<4, true>(v, sr, e0, pos0, ncols, blank);
                            else if (nb == 6) head_stage64<6, true>(v, sr, e0, pos0, ncols, blank);
                            else head_stage64_dyn<true>(v, sr, nb, e0, pos0, ncols, blank);
                        } else {
                            head_stage64_dyn<false>(v, sr, nb, e0, pos0, ncols, blank);
                        }
                    } else {
#pragma unroll
                        for (int jj = 0; jj < BNI; jj++)
                            if (jj < ncols) sts_f32(sr + 4u * jj, v[jj]);
                    }
                    __syncwarp();
                    // four rows per round, all shared-memory loads before the stores: with only four epilogue warps per SM
                    // a load -> store chain per row segment leaves the copy-out latency-bound
                    float *obase = reinterpret_cast<float *>(p.out) + seg_start + lane;
                    const uint32_t sl = smem_u32(S) + 4u * lane;
                    const bool k0 = lane < seg_len, k1 = lane + 32 < seg_len, k2 = lane + 64 < seg_len;      // seg_len <= 78
#pragma unroll 1
                    for (int rr = 0; rr < 32; rr += 4) {
                        float w[4][3];
#pragma unroll
                        for (int r = 0; r < 4; r++) {
                            const uint32_t a = sl + (uint32_t)((rr + r) * RS * 4);
                            w[r][0] = k0 ? lds_f32(a) : 0.0f;
                            w[r][1] = k1 ? lds_f32(a + 128) : 0.0f;
                            w[r][2] = k2 ? lds_f32(a + 256) : 0.0f;
                        }
#pragma unroll
                        for (int r = 0; r < 4; r++) {
                            const int mm = m0 + q * 32 + rr + r;
                            if (mm < p.M) {
                                float *o = obase + (size_t)mm * p.ldo;
                                if (k0) o[0] = w[r][0];
                                if (k1) o[32] = w[r][1];
                                if (k2) o[64] = w[r][2];
                            }
                        }
                    }
                }
            }
            __syncwarp();
        };

        // One extra (drain) round after the last tile, so that the epilogue lambda has a single call site (it is large
        // and gets inlined: three copies overflowed the instruction cache in the scores variant).
        for (int tile = blockIdx.x; tile < ntiles || pending; tile += gridDim.x) {
            const bool valid = tile < ntiles;
            const int m0 = tile * BM;
            // all MMAs of the previous tile have completed: its last accumulator may be read (by the set that owns it; a set
            // never waits on the other set's barrier, it could fall two phases behind)
            if (pending && (SETS == 1 || (int)((nit - 1) & 1) == set)) {
                mbar_wait(&acc_full[(nit - 1) & 1], ((nit - 1) >> 1) & 1);
                tc_fence_after();
            }
            // nt = -1: the previous tile's last N tile (its accumulator was awaited above), then N tiles 0 .. NT-2 of this one
            for (int nt = -1; nt < (valid ? NT - 1 : 0); nt++) {
                int em0, ent;
                uint32_t eni;
                if (nt < 0) {
                    if (!pending || (SETS > 1 && (int)((nit - 1) & 1) != set)) continue;
                    em0 = pend_m0; ent = NT - 1; eni = nit - 1;
                } else {
                    if (SETS > 1 && (int)(nit & 1) != set) { nit++; continue; }
                    if (nt == (NT > 8 ? NT - 8 : 0)) {      // next tile's x rows into L2 shortly before they are needed (G streams through L2)
                        const int mn = m0 + (int)gridDim.x * BM + r;
                        if (mn < p.M) {
                            const char *nx = reinterpret_cast<const char *>(p.x + (size_t)mn * XB_FEATURES);
#pragma unroll
                            for (int i = 0; i < 12; i++) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + i * 128));
                        }
                    }
                    mbar_wait(&acc_full[nit & 1], (nit >> 1) & 1);
                    tc_fence_after();
                    em0 = m0; ent = nt; eni = nit;
                    nit++;
                }
                epilogue(em0, ent, eni);
            }
            if (valid) {
                nit++;                                         // the last N tile is finished in the next round
                pend_m0 = m0;
            }
            pending = valid;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

}  // namespace

template <int EPI>
static int ip_launch(xb_handle *h, const void *w, int w_rows, IPParams p, cudaStream_t s) {
    // (rows, 768) 16-bit as {64 k, rows, 12 k-blocks}: one TMA lands box_kblocks K-major [box_rows x 128 B] tiles
    auto hview = [h](CUtensorMap *out, const void *base, uint64_t rows, uint32_t box_rows, uint32_t box_kblocks) {
        const uint64_t dims[3] = {64, rows, XB_FEATURES / 64}, st[2] = {XB_FEATURES * 2, 128};
        const uint32_t box[3] = {64, box_rows, box_kblocks};
        return xb_make_tmap_nd(h, out, base, 3, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_128B);
    };
    CUtensorMap tmW, tmX;
    if (int rc = hview(&tmW, w, w_rows, BNI, KPS)) return rc;
    if (int rc = hview(&tmX, p.x, (uint64_t)p.M, BM, 2)) return rc;
    p.NT = w_rows / BNI;
    const int ntiles = (p.M + BM - 1) / BM;
    const int grid = ntiles < h->num_sms ? ntiles : h->num_sms;
    constexpr int SMEM_BYTES = IPCfg<EPI>::SMEM_BYTES;
    auto kernel = inproj_kernel<EPI>;
    if (int rc = xb_smem_attr(h, kernel, SMEM_BYTES)) return rc;
    kernel<<<grid, IPCfg<EPI>::THREADS, SMEM_BYTES, s>>>(tmW, tmX, p);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

// gates (M, 3072) 16-bit = x (M, 768) . w_ih^T + bias
int xb_inproj_launch(xb_handle *h, const void *x, const void *w_ih, const float *bias, void *gates, int M, cudaStream_t s) {
    IPParams p = {};
    p.x = reinterpret_cast<const uint16_t *>(x);
    p.bias = bias;
    p.out = gates;
    p.M = M;
    p.n_valid = XB_GATES; p.ldo = XB_GATES;
    return ip_launch<IP_GATES>(h, w_ih, XB_GATES, p, s);
}

// CRF scores (M, ldo) fp32 = LinearCRFEncoder(x): the same A-stationary kernel with the head epilogue -- a CTA owns whole
// output rows, W_head (<= 2 MB) streams from L2.  w_rows = rows of the zero-padded weight (multiple of 64, <= 3072).
int xb_head_astationary_launch(xb_handle *h, const void *x, const void *w, int w_rows, const float *bias, int head_rows,
                               float *scores, int ldo, int M, int exp_out, cudaStream_t s) {
    XB_REQUIRE(h, w_rows % BNI == 0 && w_rows <= MAX_COLS && head_rows <= w_rows, "head of %d rows unsupported", head_rows);
    IPParams p = {};
    p.x = reinterpret_cast<const uint16_t *>(x);
    p.bias = bias;
    p.out = scores;
    p.M = M;
    p.n_valid = head_rows; p.ldo = ldo;
    p.n_base = h->n_base; p.expand = h->expand_blanks;
    p.scale = h->scale; p.blank = h->blank_score;
    p.exp_out = exp_out;
    return ip_launch<IP_SCORES>(h, w, w_rows, p, s);
}
