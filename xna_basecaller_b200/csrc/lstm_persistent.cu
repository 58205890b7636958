// Persistent LSTM recurrence for sm_100a: one cooperative launch runs all T steps of one layer with W_hh
// resident on chip (bonito/nn.py:176-235, RNNWrapper.forward :189-193; torch.nn.LSTM gate order i,f,g,o, zero
// initial state; a reversed layer walks time backwards by indexing instead of the reference's two flips).
//
// Decomposition.  W_hh (3072 x 768, 4.7 MB 16-bit) does not fit one SM, so it is cut into 24 tiles of 128 gate
// rows = 32 hidden units x [i,f,g,o] (rows are permuted at weight-load time, see "Epilogue layout").  The
// batch is cut into G <= 6 groups; CTA (g, j) owns tile j for group g, so 24*G <= 144 CTAs are resident, one
// per SM.
//   - the W_hh tile lives in TENSOR MEMORY for the whole kernel (128 lanes x 384 columns, the A operand of
//     tcgen05.mma), loaded once with tcgen05.st;
//   - a group is cut again into SUB sub-batches of <= NS chunks that run the recurrence independently and out
//     of phase: the serial chain of one step (h exchange through L2, TMA, MMA, cell update) is several times
//     longer than its tensor-pipe time, so the other sub-batches fill the pipe meanwhile;
//   - per step and sub-batch the CTA loads h_{t-1} (NS x 768) with one 3-D TMA box (128B swizzle; the B
//     operand), issues 48 tcgen05.mma (M=128 gate rows, N=NS chunks, K=16) into an NS-column fp32 accumulator
//     in TMEM, adds the hoisted input projection G[t] (TMA-prefetched one step ahead), applies the cell update
//     (MUFU.TANH activations) with the fp32 cell state held in registers, and writes its 32-unit slice of h_t;
//   - the 24 CTAs of a group exchange h_t through L2: after their stores the epilogue warps of a sub-batch meet
//     at a named barrier and ONE thread release-adds a per-(group, sub-batch) counter (one MEMBAR.GPU per
//     sub-batch and step: fences issued by several warps of an SM are served one after the other, eight of
//     them cost 1.4 ms per batch); the TMA producer of the sub-batch polls the counter with relaxed loads (the
//     only reader of the data is the TMA unit, issued after the poll and reading L2 directly), proxy fence,
//     next TMA load.  No CTA-wide barrier is on the per-step path.
//
// Epilogue layout.  Within a TMEM lane quarter (32 rows = 8 hidden units x 4 gates) the rows are ordered gate*8 + unit.
// tcgen05.ld.16x256b hands thread (a, b) of a warp the rows a, a+8 (and, 16 lanes further, a+16, a+24) of columns
// 8k+2b, 8k+2b+1 -- i.e. i, f, g, o of unit a for two chunks per 8 columns: every thread receives whole cells straight
// from tensor memory, no transpose and no shared-memory staging of the accumulator.
//
// Warp roles: warps 0..SUB-1 drive one sub-batch each (one elected thread: counter poll, h boxes, then the step's
// MMAs part by part as the boxes land, commit; plus the G prefetch), warp SUB allocates tensor memory, epilogue
// warps start at the next multiple of four, EW (= 8) per sub-batch (warp % 4 = TMEM lane
// quarter; the second four take the upper half of the chunk columns).  The other geometries, publish paths and
// activation forms that were measured against this one are recorded in DESIGN §4.1.
#include "xb_common.cuh"
#include "xb_ptx.cuh"
#include "xb_gemm.cuh"

using namespace xbptx;

namespace {

constexpr int TILES = 24;                  // gate tiles per group
constexpr int KCH = XB_FEATURES / 64;      // 12 K blocks of 64
constexpr int HP = 3;                      // h boxes per step: the MMAs of a box start when it lands (measured 1: 15.3,
                                           // 2: 14.9, 3: 14.8, 4: 15.4, 6: 15.4 ms per batch for the five layers)
constexpr int KPB = KCH / HP;              // K blocks per box
constexpr int D_COL = 384;                 // accumulators start after the 384 columns of W_hh
constexpr int CTR_STRIDE = 32;             // ints between counters (one 128-byte line each)
constexpr int MAX_CTRS = 64;
static_assert(MAX_CTRS * CTR_STRIDE == XB_LSTM_COUNTERS, "the handle allocates XB_LSTM_COUNTERS ints of counters");
constexpr int PREFETCH_Y = 4;              // the y rows of step s + PREFETCH_Y are prefetched into L2 at step s

// Geometry: SUB sub-batches of NS chunks per CTA, EW epilogue warps per sub-batch, two G buffers per sub-batch.
constexpr int SUB = 3;
constexpr int NS = 32;
constexpr int EW = 8;
constexpr int NB = SUB * NS;                       // chunks per group
constexpr int H_BLOCK_BYTES = NS * 64 * 2;         // one K block: NS rows x 128 B
constexpr int H_PART_BYTES = KPB * H_BLOCK_BYTES;
constexpr int H_BYTES = KCH * H_BLOCK_BYTES;
constexpr int G_BYTES = NS * 128 * 2;
constexpr int NBAR = HP + 1 + 4;                   // h_full[HP], d_full, g_full[2], g_empty[2]
constexpr int EPI_WARP0 = ((SUB + 1 + 3) / 4) * 4;
constexpr int THREADS = (EPI_WARP0 + EW * SUB) * 32;
constexpr int NC = NS * 4 / EW;                    // accumulator columns (chunks) per epilogue warp
constexpr int STAGE_BYTES = NC * 16;               // per epilogue warp: [chunk][8 units] 16-bit
constexpr int SMEM_BYTES = SUB * (H_BYTES + 2 * G_BYTES + EW * STAGE_BYTES) + 1024 /*align*/ + 1024 /*barriers*/;
static_assert(D_COL + SUB * NS <= 512, "tensor memory columns");
static_assert(NS % 16 == 0 && NS <= 48, "MMA N");
static_assert(EW % 4 == 0 && NC == 16, "epilogue split: one pair of tcgen05.ld.16x256b.x2 per warp and step");
static_assert(SUB * NBAR * 8 + 16 <= 1024, "barrier block");
static_assert(H_BLOCK_BYTES % 1024 == 0, "swizzle atom alignment");

struct PLParams {
    int T, N, reverse;
    int batch0, nbatch, G;      // batch rows [batch0, batch0 + nbatch) are split into G groups
    const uint16_t *w_hh;       // (3072, 768) 16-bit, tile-permuted rows (repack mode 4 in xb_api.cu)
    uint16_t *y;                // (T, N, 768) 16-bit output = hidden states
    int *counters;              // G * SUB counters, CTR_STRIDE ints apart, zeroed before launch
    uint16_t *save;             // training forward (SAVE kernels): (T, N, 5, 768) fp16 = activated i, f, g, o and the cell state c
};

__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// tcgen05.ld.16x256b.x2: 16 lanes x 16 columns; thread t gets rows t/4 and t/4+8, columns 8k + 2(t%4), +1:
// r[4k + {0,1}] = row t/4, r[4k + {2,3}] = row t/4 + 8  (layout checked on hardware: tools/tmem_layout_probe.cu)
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
}
template <bool SAVE>
__global__ void __launch_bounds__(THREADS, 1)
lstm_persistent_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmG, const PLParams p) {
    using X = xb16<false>;                                      // fp16 operands in both weight modes (xb_api.cu repack)
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *hbuf = smem;                                       // [SUB][H_BYTES]
    uint8_t *gbuf = smem + SUB * H_BYTES;                       // [SUB][2][G_BYTES]
    uint8_t *stage = gbuf + SUB * 2 * G_BYTES;                  // [SUB][EW][STAGE_BYTES]
    uint64_t *bars = reinterpret_cast<uint64_t *>(stage + SUB * EW * STAGE_BYTES);
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(bars + SUB * NBAR);
    auto h_full = [&](int sub, int part) { return bars + sub * NBAR + part; };
    auto d_full = [&](int sub) { return bars + sub * NBAR + HP; };
    auto g_full = [&](int sub, int q) { return bars + sub * NBAR + HP + 1 + q; };
    auto g_empty = [&](int sub, int q) { return bars + sub * NBAR + HP + 3 + q; };

    // warp index through a shuffle: tells the compiler it is warp-uniform, so the role branches below are
    // non-divergent and the epilogue shuffles need no re-convergence barriers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int g = blockIdx.x / TILES, j = blockIdx.x % TILES;
    const int T = p.T, N = p.N;
    // Groups take whole sub-batches of NS chunks (units): every sub-batch but the batch's last is full; the step time is set
    // by the chain latency, not by the number of chains per SM, so groups of two and of three sub-batches cost the same.
    const int units = (p.nbatch + NS - 1) / NS;
    const int b0 = p.batch0 + NS * (int)(((long long)g * units) / p.G);
    const int b1 = min(p.batch0 + p.nbatch, p.batch0 + NS * (int)(((long long)(g + 1) * units) / p.G));
    const int count = b1 - b0;               // <= NB valid chunks in this group
    auto sub_row0 = [&](int sub) { return b0 + sub * NS; };
    auto sub_cnt = [&](int sub) { return max(0, min(NS, count - sub * NS)); };

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmY);
        prefetch_tmap(&tmG);
        for (int sub = 0; sub < SUB; sub++) {
            for (int part = 0; part < HP; part++) mbar_init(h_full(sub, part), 1);
            mbar_init(d_full(sub), 1);
            for (int q = 0; q < 2; q++) {
                mbar_init(g_full(sub, q), 1);
                mbar_init(g_empty(sub, q), EW);
            }
        }
        fence_barrier_init();
    }
    if (warp == SUB) {
        tmem_alloc(tmem_holder, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    // W_hh tile -> tensor memory: lane = row of the tile, column c holds elements k = 2c, 2c+1
    if (warp >= EPI_WARP0 && warp < EPI_WARP0 + 4) {
        const int q = warp & 3, r = q * 32 + lane;
        const uint4 *src = reinterpret_cast<const uint4 *>(p.w_hh + ((size_t)j * 128 + r) * XB_FEATURES);
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
        for (int c0 = 0; c0 < XB_FEATURES / 2; c0 += 32) {
            uint32_t v[32];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                uint4 t4 = __ldg(src + c0 / 4 + i);
                v[4 * i] = t4.x; v[4 * i + 1] = t4.y; v[4 * i + 2] = t4.z; v[4 * i + 3] = t4.w;
            }
            tmem_st_32x32b_x32(taddr + c0, v);
        }
        tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp < SUB) {
        // ------------------------------------------------------------------ TMA producer of sub-batch `warp`
        // (elect_one, not lane == 0: the compiler must see a single, warp-uniform issuer to keep TMA / MMA
        // operands in uniform registers)
        if (elect_one()) {
            const int sub = warp;
            const int row0 = sub_row0(sub);
            const int cnt_sub = sub_cnt(sub);
            const int *ctr = p.counters + (g * SUB + sub) * CTR_STRIDE;
            uint8_t *hb = hbuf + sub * H_BYTES;
            constexpr uint32_t idesc = umma_idesc_f16(0u, 128, NS);
            const uint64_t bdesc0 = umma_desc_sw128(smem_u32(hb));
            const uint32_t dcol = tmem_base + D_COL + sub * NS;
            if (cnt_sub > 0) {
                mbar_expect_tx(g_full(sub, 0), G_BYTES);
                tma_load_2d(gbuf + (sub * 2) * G_BYTES, &tmG, g_full(sub, 0), j * 128, (p.reverse ? T - 1 : 0) * N + row0);
            }
            for (int s = 0; s < (cnt_sub > 0 ? T : 0); s++) {      // an empty sub-batch (a short last group) has no chain
                const int t = p.reverse ? T - 1 - s : s;
                if (s + 1 < T) {                 // input projection of the next step, one step ahead
                    const int sn = s + 1, q = sn & 1, u = sn >> 1;
                    const int tn = p.reverse ? T - 1 - sn : sn;
                    if (u >= 1) mbar_wait(g_empty(sub, q), (u - 1) & 1);
                    mbar_expect_tx(g_full(sub, q), G_BYTES);
                    tma_load_2d(gbuf + (sub * 2 + q) * G_BYTES, &tmG, g_full(sub, q), j * 128, tn * N + row0);
                }
                if (s + PREFETCH_Y < T) {
                    // bring the y rows this sub-batch will write PREFETCH_Y steps from now into L2 (one row per CTA and
                    // sub-batch, round robin over the group's tiles): a 16-byte store to a line that is not resident is only
                    // acknowledged after the line was fetched from HBM, which is what the release below waits for.  At most
                    // two rows (NS <= 2 * TILES): unrolled, the loop held five more registers than the kernel needs elsewhere.
                    const int t2 = p.reverse ? T - 1 - (s + PREFETCH_Y) : s + PREFETCH_Y;
#pragma unroll 1
                    for (int r = j; r < cnt_sub; r += TILES)
                        prefetch_l2_bulk(p.y + ((size_t)t2 * N + row0 + r) * XB_FEATURES, XB_FEATURES * 2);
                }
                if (s > 0) {
                    const int tp = p.reverse ? t + 1 : t - 1;
                    const int need = TILES * EW * s;         // every epilogue warp of the group has published step s-1
                    // relaxed spin (an acquire load per iteration costs a CCTL.IVALL each time), then ONE acquire load of
                    // the counter once it has been seen at its target: that load synchronises with the producers'
                    // red.release (PTX memory model: a relaxed load alone does not), the proxy fence then orders the
                    // TMA unit's reads of h behind it
                    while (ld_relaxed_gpu(ctr) < need) {
                    }
                    (void)ld_acquire_gpu(ctr);
                    fence_proxy_async_global();
                    // h_{t-1} of the sub-batch: HP boxes {64 k, NS chunks, KPB k-blocks}, each landing as KPB
                    // swizzled [NS x 128 B] K-major tiles on its own mbarrier
#pragma unroll
                    for (int part = 0; part < HP; part++) {
                        mbar_expect_tx(h_full(sub, part), H_PART_BYTES);
                        tma_load_3d(hb + part * H_PART_BYTES, &tmY, h_full(sub, part), 0, tp * N + row0, part * KPB);
                    }
                    // ... and the MMAs of the step, part by part as the boxes land (blocking try_wait: ~60 cycles from
                    // completion to wake-up; an earlier single MMA warp scanning all sub-batches with test_wait paid
                    // ~150 cycles per probe and could not keep up with more than one box per step)
#pragma unroll
                    for (int part = 0; part < HP; part++) {
                        mbar_wait(h_full(sub, part), (s - 1) & 1);
                        tc_fence_after();
#pragma unroll
                        for (int kk = 0; kk < KPB * 4; kk++) {
                            const int kc = kk >> 2, k = kk & 3;
                            mma_f16_ts(dcol, tmem_base + part * (KPB * 32) + kk * 8,
                                       bdesc0 + (uint64_t)((part * H_PART_BYTES + kc * H_BLOCK_BYTES + k * 32) >> 4), idesc,
                                       (part | kk) != 0);
                        }
                    }
                    mma_commit(d_full(sub));
                }
            }
        }
    } else if (warp >= EPI_WARP0) {
        // ------------------------------------------------------------------ epilogue (EW warps per sub-batch: warp % 4 =
        // TMEM lane quarter; the second four take the upper half of the chunk columns)
        constexpr int CELLS = NC / 4;
        const int ew = (warp - EPI_WARP0) % EW, sub = (warp - EPI_WARP0) / EW, q = warp & 3;
        const int col0 = (ew >> 2) * NC;                     // first chunk column of this warp
        const int gt = lane & 3, ul = lane >> 2;             // gate held after the TMEM load; unit within the warp
        const int unit = q * 8 + ul;                         // unit within the tile
        const int row0 = sub_row0(sub);
        const int cnt = sub_cnt(sub);                            // valid chunks of this sub-batch (<= NS)
        // h is published through generic stores + red.release.  Publishing a full sub-batch's tile with one TMA tensor store
        // was measured and removed: with a release on the counter it was as fast as this route (14.1 ms per batch); with a
        // relaxed add it was 8-10 % faster (12.5-13.1 ms), but then nothing orders the tile's writes before the counter in
        // the PTX memory model.
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + D_COL + sub * NS + col0;
        int *ctr = p.counters + (g * SUB + sub) * CTR_STRIDE;
        float cst[CELLS];
#pragma unroll
        for (int i = 0; i < CELLS; i++) cst[i] = 0.0f;

        for (int s = 0; s < (cnt > 0 ? T : 0); s++) {
            const int t = p.reverse ? T - 1 - s : s;
            const uint16_t *Gs = reinterpret_cast<const uint16_t *>(gbuf + (sub * 2 + (s & 1)) * G_BYTES);
            // Accumulator -> registers with tcgen05.ld.16x256b: thread (a = lane/4, b = lane%4) receives rows a, a+8 (first
            // load) and a+16, a+24 (second load, 16 lanes further) of columns 8k+2b, 8k+2b+1.  The rows of a lane quarter are
            // ordered gate*8 + unit, so those four rows are i, f, g, o of unit a: the load itself delivers whole cells
            // (an earlier version read one row per thread and transposed with 16 shuffles per thread: 580 cycles).
            // The input projection of the step arrived a step ago: fetch it from shared memory BEFORE waiting for the
            // accumulator, so only the adds remain on the serial chain.
            // cell m of the thread: chunk 8*(m/2) + 2b + m%2 (relative to col0), unit ul
            mbar_wait(g_full(sub, s & 1), (s >> 1) & 1);
            float pre[CELLS][4];
#pragma unroll
            for (int m = 0; m < CELLS; m++) {
                const int ch = 8 * (m >> 1) + 2 * gt + (m & 1);
                const uint2 graw = *reinterpret_cast<const uint2 *>(Gs + (col0 + ch) * 128 + unit * 4);
                const float2 g01 = X::unpack(graw.x), g23 = X::unpack(graw.y);
                pre[m][0] = g01.x; pre[m][1] = g01.y; pre[m][2] = g23.x; pre[m][3] = g23.y;
            }
            if (s > 0) {
                uint32_t lo[NC / 2], hi[NC / 2];
                mbar_wait(d_full(sub), (s - 1) & 1);
                tc_fence_after();
                tmem_ld_16x256b_x2(taddr, lo);
                tmem_ld_16x256b_x2(taddr + (16u << 16), hi);
                tmem_ld_wait();
                tc_fence_before();
#pragma unroll
                for (int m = 0; m < CELLS; m++) {
                    const int k4 = 4 * (m >> 1), wi = m & 1;
                    pre[m][0] += __uint_as_float(lo[k4 + wi]);
                    pre[m][1] += __uint_as_float(lo[k4 + 2 + wi]);
                    pre[m][2] += __uint_as_float(hi[k4 + wi]);
                    pre[m][3] += __uint_as_float(hi[k4 + 2 + wi]);
                }
            }
            // phase B: c' = sig(f) c + sig(i) tanh(g), h = sig(o) tanh(c'), written stage by stage over all cells so
            // that the MUFU latencies overlap.
            float hout[CELLS];
            float sv[SAVE ? 5 : 1][CELLS];           // training forward: what BPTT needs of this step
            // Five MUFU.TANH per cell (sigmoid(x) = 0.5 tanh(0.5 x) + 0.5) and a dozen FMAs: a third of the instructions
            // of the exp/rcp form (7 MUFU + ~45 FP ops per cell), which was measured and removed.  tanh.approx.f32 has
            // ~2^-11 relative error, the size of the fp16 rounding of h.
#pragma unroll
            for (int i = 0; i < CELLS; i++) {
                const float si = fmaf(tanh_approx(0.5f * pre[i][0]), 0.5f, 0.5f);
                const float sf = fmaf(tanh_approx(0.5f * pre[i][1]), 0.5f, 0.5f);
                const float tg = tanh_approx(pre[i][2]);
                const float so = fmaf(tanh_approx(0.5f * pre[i][3]), 0.5f, 0.5f);
                const float cn = fmaf(sf, cst[i], si * tg);
                cst[i] = cn;
                hout[i] = so * tanh_approx(cn);
                if (SAVE) { sv[0][i] = si; sv[SAVE ? 1 : 0][i] = sf; sv[SAVE ? 2 : 0][i] = tg; sv[SAVE ? 3 : 0][i] = so; sv[SAVE ? 4 : 0][i] = cn; }
            }
            // h slice of the warp (NS chunks x 8 units) through a private 16 B-per-chunk staging row: one 16-byte global
            // store per chunk instead of eight 2-byte ones
            constexpr int ST_PITCH = 8;                          // 16-bit elements between consecutive chunks
            // explicit shared-memory instructions: behind the casts the compiler falls back to generic loads / stores
            const uint32_t st_s = smem_u32(stage + (sub * EW + ew) * STAGE_BYTES);
#pragma unroll
            for (int i = 0; i < CELLS; i++) {
                typename X::T hv = X::from(hout[i]);
                sts_u16(st_s + 2u * ((8 * (i >> 1) + 2 * gt + (i & 1)) * ST_PITCH + ul), *reinterpret_cast<uint16_t *>(&hv));
            }
            __syncwarp();
            if (lane < NC && col0 + lane < cnt)
                *reinterpret_cast<uint4 *>(p.y + ((size_t)t * N + row0 + col0 + lane) * XB_FEATURES + j * 32 + q * 8) =
                    lds_v4(st_s + 2u * (lane * ST_PITCH));
            // one release per sub-batch and step instead of one per warp (MEMBAR.GPU instances of one SM appear to
            // be served one at a time; the per-warp release was measured and removed): the sub-batch's warps meet at a
            // named barrier, one thread publishes
            named_bar_sync(1 + sub, EW * 32);
            if (ew == 0 && lane == 0)
                red_release_gpu_add(ctr, EW);                 // cumulative over the barrier: all the sub-batch's stores
            if (lane == 0) mbar_arrive(g_empty(sub, s & 1));
            // Training forward: i, f, g, o, c of the step through the same private staging rows -> (T, N, 5, 768) fp16.
            // AFTER h has been published: these stores feed the backward pass, not the next step, and in front of the release
            // they sat on the step-to-step chain (five staging rounds, and the release's fence waits for every store before it).
            if (SAVE) {
#pragma unroll
                for (int qn = 0; qn < 5; qn++) {
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < CELLS; i++) {
                        const __half hv = __float2half_rn(sv[SAVE ? qn : 0][i]);
                        sts_u16(st_s + 2u * ((8 * (i >> 1) + 2 * gt + (i & 1)) * ST_PITCH + ul), *reinterpret_cast<const uint16_t *>(&hv));
                    }
                    __syncwarp();
                    if (lane < NC && col0 + lane < cnt)
                        *reinterpret_cast<uint4 *>(p.save + (((size_t)t * N + row0 + col0 + lane) * 5 + qn) * XB_FEATURES + j * 32 + q * 8) =
                            lds_v4(st_s + 2u * (lane * ST_PITCH));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == SUB) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

template <bool SAVE>
int launch(xb_handle *h, int layer, void *y_tnc, int T, int N, int reverse, cudaStream_t s, void *save) {
    CUtensorMap tmY, tmG;
    {       // y (T*N, 768) as {64 k, rows, 12 k-blocks}: one TMA lands KPB K-major [NS x 128 B] tiles
        const uint64_t dims[3] = {64, (uint64_t)T * N, XB_FEATURES / 64}, st[2] = {XB_FEATURES * 2, 128};
        const uint32_t box[3] = {64, NS, KPB};
        if (int rc = xb_make_tmap_nd(h, &tmY, y_tnc, 3, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    {       // gates (T*N, 3072), 128 x NS boxes, not swizzled
        const uint64_t dims[2] = {XB_GATES, (uint64_t)T * N}, st[1] = {XB_GATES * 2};
        const uint32_t box[2] = {128, NS};
        if (int rc = xb_make_tmap_nd(h, &tmG, h->gates, 2, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return rc;
    }
    const int max_groups = h->num_sms / TILES;                 // 6 on a 148-SM B200
    if (max_groups < 1)
        return xb_fail(h, XB_ERR_UNSUPPORTED, "the persistent LSTM needs %d co-resident CTAs, the device has %d SMs", TILES, h->num_sms);
    const int block_cap = max_groups * NB;
    auto fn = lstm_persistent_kernel<SAVE>;
    if (int rc = xb_smem_attr(h, fn, SMEM_BYTES)) return rc;
    for (int batch0 = 0; batch0 < N; batch0 += block_cap) {
        PLParams p;
        p.T = T; p.N = N; p.reverse = reverse;
        p.batch0 = batch0;
        p.nbatch = (N - batch0 < block_cap) ? N - batch0 : block_cap;
        p.G = (p.nbatch + NB - 1) / NB;
        p.w_hh = reinterpret_cast<const uint16_t *>(h->lstm[layer].w_hh);
        p.y = reinterpret_cast<uint16_t *>(y_tnc);
        p.counters = h->lstm_counters;
        p.save = reinterpret_cast<uint16_t *>(save);
        XB_CUDA(h, cudaMemsetAsync(h->lstm_counters, 0, XB_LSTM_COUNTERS * sizeof(int), s));
        void *args[] = {(void *)&tmY, (void *)&tmG, (void *)&p};
        XB_CUDA(h, cudaLaunchCooperativeKernel((const void *)fn, dim3(p.G * TILES), dim3(THREADS), args, SMEM_BYTES, s));
        h->launches++;
    }
    return XB_OK;
}

}  // namespace

// Recurrent part of one LSTM layer.  h->gates must already hold the input projection (T*N, 3072) with the
// columns of every 128-wide tile ordered [unit][i,f,g,o] (weight repack mode 3 in xb_api.cu).
// save != nullptr: the training forward, which also stores (T, N, 5, 768) fp16 = i, f, g, o, c for the backward pass
int xb_lstm_recurrence_persistent(xb_handle *h, int layer, void *y_tnc, int T, int N, int reverse, cudaStream_t s, void *save) {
    if (save) return launch<true>(h, layer, y_tnc, T, N, reverse, s, save);
    return launch<false>(h, layer, y_tnc, T, N, reverse, s, nullptr);
}
