// CTC-CRF decode in the LINEAR domain for sm_100a: posteriors (Log semiring) and max-marginal Viterbi labels
// (Max semiring over log(posterior + 1e-8)) without a single logarithm and with one exponential per edge.
//
// Reference semantics: bonito/crf/model.py:41-46 (logZ boundary conditions alpha_0 = beta_T = 0), the inherited
// seqdist posteriors (restated in oracle/seqdist_restated.py), :92-95 (viterbi = posteriors(Max).argmax % NZ),
// :215-218 (decode_batch: log(posteriors + 1e-8) -> viterbi), :97-100 and bonito/crf/basecall.py:56-76 (letters,
// left-packed rows).  The arithmetic contract -- operation order, reduction trees, the exact exp -- is the one written
// above xbo_crf_decode_lin_range in oracle/c/crf_exact.c; kernels and checker must stay in lock step because the
// tests demand bit-equal labels.
//
// Why linear.  In the log domain every state costs NZ exps + one log per step and sweep, and the softmax over the
// C*NZ edges of a step another exp + NZ logs: the round-1 sweeps were issue-bound at 15% of the HBM roofline.  Here
//   E = exp(M)                              one exact exp per edge (none at all when the fused head already wrote E),
//   Log semiring  -> sums of products,      Max semiring over log(p + 1e-8) -> max of products of (p + 1e-8),
// and every state vector is rescaled by a power of two taken from its own maximum (exact), so nothing leaves the fp32
// range.  Against a float64 evaluation the posteriors are 1000x closer than the log-domain fp32 formulation
// (1.5e-7 vs 1.6e-4 at T = 800: log-domain alphas grow to ~1e3, where one ulp is 6e-5).
//
// Three sweeps, one CTA per sequence, one thread per state, score rows and state vectors through a ring of TMA bulk
// copies (one elected thread issues them, mbarrier completion), ONE CTA barrier per step:
//   1 crf_lin_alpha     forward:  a_hat (T+1,N,C)
//   2 crf_lin_backward  backward: b_hat (T+1,N,C), the per-step normaliser tot (T,N), and -- one step behind, because it
//                       needs 1/tot of the step -- the Max-semiring beta over P = p + 1e-8: bm_hat (T+1,N,C)
//   3 crf_lin_viterbi   forward:  P again from E, a_hat, b_hat, tot (same operands in the same order: same bits),
//                       Max-semiring alpha, arg-max edge -> label -> letters -> left-packed row; optional posteriors out.
// HBM traffic per (t, sequence): 3 reads of the score row S = 4*C*NZ bytes + 7 state vectors of 4*C bytes, against
// the 2*S + 1 that SURVEY 8(d) counts as algorithmic.
#include "xb_common.cuh"
#include "xb_exact_math.h"
#include "crf_lattice.cuh"
#include "xb_ptx.cuh"

using namespace xbcrf;

namespace {

// maximum of non-negative floats over a warp: their bit patterns are ordered like the values
__device__ __forceinline__ float warp_max_pos(float v) {
    return __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(v)));
}
template <int W> __device__ __forceinline__ float red_max(const float *red) {
    float m = red[0];
#pragma unroll
    for (int i = 1; i < W; i++) m = fmaxf(m, red[i]);
    return m;
}
template <bool LIN> __device__ __forceinline__ float edge_E(float m) { return LIN ? m : xb_score_exp(m); }

// ---- the row ring: TMA bulk copies (cp.async.bulk global -> shared, mbarrier completion) -------------------------
// One elected thread moves every score row and state vector of a step with a handful of bulk copies; the other
// threads issue no copy instructions at all (the 8-byte cp.async ring of round 1 cost every thread three LDGSTS + their
// address arithmetic per step and kept the load/store pipe as busy as the arithmetic).
// Bulk copies need 16-byte aligned addresses and sizes.  Score rows of the 5-letter alphabet are 3000 bytes, so every
// other row starts 8 bytes off: such a row is copied from its aligned-down address (8 bytes more, the same constant
// size for both phases) and read at the matching offset inside its slot.  State vectors live in handle workspace with a
// pitch of VP = NT + 4 floats, 16-byte aligned; slot NT of a b_hat vector carries the step's normaliser.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(xbptx::smem_u32(bar)) : "memory");
}

template <int NB, int SL> struct Ring {
    using L = Lat<NB, SL>;
    static constexpr int ROWB = L::S * 4;                          // bytes of one score row
    static constexpr bool PHASED = (ROWB % 16) != 0;               // rows alternate between phase 0 and phase 8
    static_assert(ROWB % 8 == 0, "score rows are at least 8-byte aligned");
    static constexpr int ROW_COPY = PHASED ? ROWB + 8 : ROWB;      // bytes per row copy (multiple of 16)
    static constexpr int ROWF = ROW_COPY / 4;                      // floats per row slot
    static constexpr int VP = L::NT + 4;                           // state vector pitch (floats)
    static constexpr int VECB = VP * 4;
    // float offset of row `rid` (= t * N + n) inside its slot
    static __device__ __forceinline__ int phase(size_t rid) { return PHASED ? (int)(rid & 1) * 2 : 0; }
    // Arm the slot's barrier for the row + `extra_tx` bytes of state vectors and issue the row copy (elected thread).
    // total_rows guards the 8 bytes past the tensor's end: the last row of the tensor in phase 0 is copied 8 bytes short and
    // its tail moved by hand -- BEFORE the arrive, whose release orders that generic store ahead of the consumers' wait.
    static __device__ __forceinline__ void fetch_row(float *slot, const float *scores, size_t rid, size_t total_rows,
                                                     uint64_t *bar, uint32_t extra_tx) {
        const char *src = reinterpret_cast<const char *>(scores) + rid * ROWB;
        if (PHASED && !(rid & 1) && rid + 1 == total_rows) {
            const float2 tail = *reinterpret_cast<const float2 *>(src + ROWB - 8);
            *reinterpret_cast<float2 *>(reinterpret_cast<char *>(slot) + ROWB - 8) = tail;
            xbptx::mbar_expect_tx(bar, ROWB - 8 + extra_tx);
            bulk_g2s(xbptx::smem_u32(slot), src, ROWB - 8, bar);
            return;
        }
        xbptx::mbar_expect_tx(bar, ROW_COPY + extra_tx);
        bulk_g2s(xbptx::smem_u32(slot), (PHASED && (rid & 1)) ? src - 8 : src, ROW_COPY, bar);
    }
};

// Thread roles of the three sweeps: W = NT / 32 COMPUTE warps (one thread per state; they meet at named barrier 1 once per
// step to exchange the state vector) and one SERVICE warp that runs ahead on its own: it waits for a ring slot to be
// released (mbarrier `empty`, one arrival per compute warp), issues the bulk copies of the row D-1 steps ahead, and -- in
// the Viterbi sweep -- reduces the per-warp arg-max candidates of a step to its label.  Keeping the copy issue and that
// serial reduction out of the compute warps took a third off the per-step latency (the whole CTA used to wait at the
// barrier for the one warp that had done them).
template <int NB, int SL> struct Roles {
    using L = Lat<NB, SL>;
    static constexpr int NT = L::NT, W = L::W, NTT = NT + 32;
};
__device__ __forceinline__ void compute_bar(int nt) { asm volatile("bar.sync 1, %0;" ::"r"(nt) : "memory"); }
// The service warp runs D-1 steps ahead and spends most of its life waiting for a slot to be released: it must not burn
// issue slots doing so (a bare try_wait loop re-issues every few dozen cycles; ncu showed it executing a third of the
// CTA's instructions), and nothing is lost if it notices a free slot a few hundred nanoseconds late.
__device__ __forceinline__ void service_wait(uint64_t *bar, uint32_t parity) {
    while (!xbptx::mbar_try_wait(bar, parity)) __nanosleep(256);
}

// --------------------------------------------------------------------------------------------------
// Sweep 1, forward: a_hat_0 = 1;  u_{t+1}[c] = fma-chain_k E_t[c,k] * a_hat_t[src(c,k)];  a_hat = u * scale(max u).
// The scale of a vector is known one barrier after the vector, so a_hat_t is applied (and stored) at step t.
template <int NB, int SL, bool LIN>
__global__ void __launch_bounds__(Lat<NB, SL>::NT + 32)
crf_lin_alpha_kernel(const float *__restrict__ scores, int T, int N, float *__restrict__ alpha_out) {
    using L = Lat<NB, SL>;
    using R = Ring<NB, SL>;
    constexpr int C = L::C, NZ = L::NZ, NT = L::NT, W = L::W, D = L::D;
    extern __shared__ __align__(128) float smem[];
    float *ring = smem;                      // D * ROWF
    float *u = ring + D * R::ROWF;           // 2 * NT
    float *red = u + 2 * NT;                 // 2 * W
    uint64_t *full = reinterpret_cast<uint64_t *>((reinterpret_cast<uintptr_t>(red + 2 * W) + 7) & ~uintptr_t(7));   // D + D barriers
    uint64_t *empty = full + D;
    const int n = blockIdx.x, c = threadIdx.x, lane = c & 31, w = c >> 5;
    const size_t total_rows = (size_t)T * N;
    if (c == NT) {
        for (int j = 0; j < D; j++) { xbptx::mbar_init(&full[j], 1); xbptx::mbar_init(&empty[j], W); }
        xbptx::fence_barrier_init();
    }
    if (c < NT) {
        u[c] = c < C ? 1.0f : 0.0f;
        if (lane == 0) red[w] = 1.0f;
    }
    __syncthreads();
    if (w == W) {                            // ---------------- service warp
        if (lane == 0) {
            auto fetch = [&](int r) {
                const size_t rid = (size_t)r * N + n;
                R::fetch_row(ring + (r % D) * R::ROWF, scores, rid, total_rows, &full[r % D], 0);
            };
            for (int j = 0; j < D - 1 && j < T; j++) fetch(j);
            for (int t = 0; t + D - 1 < T; t++) {
                if (t > 0) service_wait(&empty[(t - 1) % D], ((t - 1) / D) & 1);
                fetch(t + D - 1);
            }
        }
        return;
    }
    const bool act = c < C;
    int src[NZ];
    src[0] = act ? c : 0;
#pragma unroll
    for (int k = 1; k < NZ; k++) src[k] = act ? (k - 1) * L::NP + c / NB : 0;
    float *aout = alpha_out + (size_t)n * R::VP + c;
    const size_t arow = (size_t)N * R::VP;
    float uprev = 1.0f;
    for (int t = 0; t < T; t++) {
        const int slot = t % D;
        xbptx::mbar_wait(&full[slot], (t / D) & 1);
        compute_bar(NT);
        const float sc = xb_pow2_scale(red_max<W>(red + (t & 1) * W));
        const float *M = ring + slot * R::ROWF + R::phase((size_t)t * N + n) + c * NZ;
        const float *uc = u + (t & 1) * NT;
        float acc = 0.0f;
        if (act) {
            float e[NZ];
#pragma unroll
            for (int k = 0; k < NZ; k++) e[k] = edge_E<LIN>(M[k]);
            *aout = XB_MUL(uprev, sc);
            acc = XB_MUL(e[0], XB_MUL(uc[src[0]], sc));
#pragma unroll
            for (int k = 1; k < NZ; k++) acc = XB_FMA(e[k], XB_MUL(uc[src[k]], sc), acc);
            u[((t + 1) & 1) * NT + c] = acc;
            uprev = acc;
        }
        __syncwarp();
        if (lane == 0) xbptx::mbar_arrive(&empty[slot]);
        aout += arow;
        const float wm = warp_max_pos(acc);
        if (lane == 0) red[((t + 1) & 1) * W + w] = wm;
    }
    compute_bar(NT);
    if (act) *aout = XB_MUL(uprev, xb_pow2_scale(red_max<W>(red + (T & 1) * W)));
}

// --------------------------------------------------------------------------------------------------
// Sweep 2, backward.  Thread s is the SOURCE state of its NZ outgoing edges (stay, then the moves j = 0..NB-1 into
// state (s % NP) * NB + j through edge k = 1 + s / NP).  Iteration i handles the Log step t = T-1-i:
//     w_e = E_t[e] * b_hat_{t+1}[dst_e];  u_t[s] = sum_e w_e;  x_e = a_hat_t[s] * w_e;  tot_t = tree_sum_s(sum_e x_e)
// and, one step behind (1 / tot_{t+1} is only known after this iteration's barrier), the Max step t+1:
//     um_{t+1}[s] = max_e (x_e(t+1) / tot_{t+1} + 1e-8) * bm_hat_{t+2}[dst_e]
// with the x_e of the previous iteration held in registers.  tot_t is stored in slot NT of the b_hat_{t+1} vector.
template <int NB, int SL, bool LIN>
__global__ void __launch_bounds__(Lat<NB, SL>::NT + 32)
crf_lin_backward_kernel(const float *__restrict__ scores, const float *__restrict__ alpha, int T, int N,
                        float *__restrict__ beta_out, float *__restrict__ bmax_out) {
    using L = Lat<NB, SL>;
    using R = Ring<NB, SL>;
    constexpr int C = L::C, NZ = L::NZ, NT = L::NT, W = L::W, D = L::D;
    extern __shared__ __align__(128) float smem[];
    float *ring = smem;                      // D * ROWF
    float *ringA = ring + D * R::ROWF;       // D * VP: a_hat_t
    float *ub = ringA + D * R::VP;           // 2 * NT
    float *um = ub + 2 * NT;                 // 2 * NT
    float *redb = um + 2 * NT;               // 2 * W
    float *redm = redb + 2 * W;              // 2 * W
    float *part = redm + 2 * W;              // 2 * W
    uint64_t *full = reinterpret_cast<uint64_t *>((reinterpret_cast<uintptr_t>(part + 2 * W) + 7) & ~uintptr_t(7));   // D + D barriers
    uint64_t *empty = full + D;
    const int n = blockIdx.x, s = threadIdx.x, lane = s & 31, w = s >> 5;
    const size_t total_rows = (size_t)T * N;
    const size_t vrow = (size_t)N * R::VP;
    if (s == NT) {
        for (int j = 0; j < D; j++) { xbptx::mbar_init(&full[j], 1); xbptx::mbar_init(&empty[j], W); }
        xbptx::fence_barrier_init();
    }
    // buffers are read at parity q = i & 1 and written at q ^ 1; the Max recursion starts at iteration 1 (parity 1)
    if (s < NT) {
        ub[s] = s < C ? 1.0f : 0.0f;
        um[NT + s] = s < C ? 1.0f : 0.0f;
        if (lane == 0) { redb[w] = 1.0f; redm[W + w] = 1.0f; }
    }
    __syncthreads();
    if (w == W) {                            // ---------------- service warp
        if (lane == 0) {
            const float *abase = alpha + (size_t)n * R::VP;
            auto fetch = [&](int r) {        // iteration r: score row and a_hat of step T-1-r
                const int t = T - 1 - r, slot = r % D;
                const size_t rid = (size_t)t * N + n;
                R::fetch_row(ring + slot * R::ROWF, scores, rid, total_rows, &full[slot], R::VECB);
                bulk_g2s(xbptx::smem_u32(ringA + slot * R::VP), abase + (size_t)t * vrow, R::VECB, &full[slot]);
            };
            for (int j = 0; j < D - 1 && j < T; j++) fetch(j);
            for (int i = 0; i + D - 1 < T; i++) {
                if (i > 0) service_wait(&empty[(i - 1) % D], ((i - 1) / D) & 1);
                fetch(i + D - 1);
            }
        }
        return;
    }
    const bool act = s < C;
    const int kk = act ? 1 + s / L::NP : 1, cb = act ? (s % L::NP) * NB : 0;
    int eidx[NZ], dst[NZ];               // edge index into the row / destination state, e = 0 stay, 1 + j moves
    eidx[0] = (act ? s : 0) * NZ; dst[0] = act ? s : 0;
#pragma unroll
    for (int j = 0; j < NB; j++) { eidx[1 + j] = (cb + j) * NZ + kk; dst[1 + j] = cb + j; }

    float *bout = beta_out + (size_t)T * vrow + (size_t)n * R::VP + s;        // b_hat_{t+1}, written at iteration i
    float *mout = bmax_out + (size_t)T * vrow + (size_t)n * R::VP + s;        // bm_hat_{t+2}, written at iteration i >= 1
    float ubprev = 1.0f, umprev = 1.0f;
    float x[NZ];
#pragma unroll
    for (int e = 0; e < NZ; e++) x[e] = 0.0f;
    for (int i = 0; i <= T; i++) {
        const int t = T - 1 - i, q = i & 1, slot = i % D;
        if (i < T) xbptx::mbar_wait(&full[slot], (i / D) & 1);
        compute_bar(NT);
        const float sb = xb_pow2_scale(red_max<W>(redb + q * W));
        float ev[NZ], bv[NZ], a = 0.0f;
        if (i < T && act) {                  // everything this step needs from the ring slot, then release it
            const float *M = ring + slot * R::ROWF + R::phase((size_t)t * N + n);
#pragma unroll
            for (int e = 0; e < NZ; e++) ev[e] = edge_E<LIN>(M[eidx[e]]);
            a = ringA[slot * R::VP + s];
        }
        if (i < T) {
            __syncwarp();
            if (lane == 0) xbptx::mbar_arrive(&empty[slot]);
        }
        if (act) *bout = XB_MUL(ubprev, sb);
        if (i >= 1) {                        // Max step t+1 with the x of the previous iteration
            float tot = part[q * W];
#pragma unroll
            for (int j = 1; j < W; j++) tot = XB_ADD(tot, part[q * W + j]);
            if (s == 0) bout[vrow + NT] = tot;                   // slot NT of b_hat_{t+2}: the normaliser of step t+1
            const float inv = XB_RCP(tot);
            const float sm = xb_pow2_scale(red_max<W>(redm + q * W));
            const float *mc = um + q * NT;
            float best = 0.0f;
            if (act) {
                *mout = XB_MUL(umprev, sm);
#pragma unroll
                for (int e = 0; e < NZ; e++) {
                    const float v = XB_MUL(XB_ADD(XB_MUL(x[e], inv), XB_POST_EPS), XB_MUL(mc[dst[e]], sm));
                    best = (e == 0) ? v : fmaxf(best, v);
                }
                um[(q ^ 1) * NT + s] = best;
                umprev = best;
            }
            mout -= vrow;
            const float wm = warp_max_pos(best);
            if (lane == 0) redm[(q ^ 1) * W + w] = wm;
        }
        bout -= vrow;
        if (i < T) {                         // Log step t
            const float *bc = ub + q * NT;
            float su = 0.0f, sx = 0.0f;
            if (act) {
#pragma unroll
                for (int e = 0; e < NZ; e++) bv[e] = XB_MUL(bc[dst[e]], sb);
#pragma unroll
                for (int e = 0; e < NZ; e++) {
                    const float we = XB_MUL(ev[e], bv[e]);
                    x[e] = XB_MUL(a, we);
                    su = (e == 0) ? we : XB_ADD(su, we);
                    sx = (e == 0) ? x[e] : XB_ADD(sx, x[e]);
                }
                ub[(q ^ 1) * NT + s] = su;
                ubprev = su;
            }
            const float wm = warp_max_pos(su);
            const float ws = warp_sum_tree(sx);
            if (lane == 0) { redb[(q ^ 1) * W + w] = wm; part[(q ^ 1) * W + w] = ws; }
        }
    }
}

// --------------------------------------------------------------------------------------------------
// Sweep 3, forward, Max semiring over P.  Thread c is the DESTINATION state of its NZ incoming edges.
//     P_k = a_hat_t[src_k] * (E_t[c,k] * b_hat_{t+1}[c]) / tot_t + 1e-8        (the bits sweep 2 produced)
//     v_k = P_k * am_hat_t[src_k];  um_{t+1}[c] = max_k v_k;  candidate v_k * bm_hat_{t+1}[c]
// arg-max over the flat edge index (first index on ties) -> label = edge % NZ -> letters -> left-packed row.
template <int NB, int SL, bool LIN, bool POST>
__global__ void __launch_bounds__(Lat<NB, SL>::NT + 32)
crf_lin_viterbi_kernel(const float *__restrict__ scores, const float *__restrict__ alpha, const float *__restrict__ beta,
                       const float *__restrict__ bmax, int T, int N,
                       int8_t *__restrict__ labels_out, int8_t *__restrict__ seq_out, int8_t *__restrict__ qs_out,
                       int32_t *__restrict__ lens_out, float *__restrict__ post_out, Alphabet abc) {
    using L = Lat<NB, SL>;
    using R = Ring<NB, SL>;
    constexpr int C = L::C, NZ = L::NZ, S = L::S, NT = L::NT, W = L::W, D = L::D, NTT = NT + 32;
    extern __shared__ __align__(128) float smem[];
    float *ring = smem;                      // D * ROWF
    float *ringA = ring + D * R::ROWF;       // D * VP: a_hat_t (whole vector: sources)
    float *ringB = ringA + D * R::VP;        // D * VP: b_hat_{t+1} (+ tot_t in slot NT)
    float *ringM = ringB + D * R::VP;        // D * VP: bm_hat_{t+1}
    float *am = ringM + D * R::VP;           // 2 * NT
    float *redm = am + 2 * NT;               // 2 * W
    float *bval = redm + 2 * W;              // D * W: per-warp arg-max candidates of the last D steps
    int *bidx = reinterpret_cast<int *>(bval + D * W);      // D * W
    uint64_t *full = reinterpret_cast<uint64_t *>((reinterpret_cast<uintptr_t>(bidx + D * W) + 7) & ~uintptr_t(7));   // 3 * D barriers
    uint64_t *empty = full + D, *cand = empty + D;
    int *scan = reinterpret_cast<int *>(cand + D);          // NTT + 1
    int8_t *lab = reinterpret_cast<int8_t *>(scan + NTT + 1);   // T
    // POST: two staged posterior rows.  A thread owns NZ consecutive floats of a row (28-byte lane stride for NZ = 7): written
    // straight to global memory every store instruction fills a sliver of ~28 sectors.  The row is staged here instead and
    // leaves one step later, after the barrier the next step needs anyway, as whole 128-byte segments.
    // Only for the larger lattices (XY: 6 KB rows, 1024 sequences): on X (3 KB rows) the sweep is issue-bound and the extra
    // shared-memory round trip costs more than the slivers (measured 1.04 against 0.82 ms at N = 512).
    constexpr bool PSTAGE = POST && L::S >= 1024;
    float *pst = PSTAGE ? reinterpret_cast<float *>(lab + ((T + 15) / 16) * 16) : nullptr;      // 2 * S
    const int n = blockIdx.x, c = threadIdx.x, lane = c & 31, w = c >> 5;
    const size_t total_rows = (size_t)T * N;
    const size_t vrow = (size_t)N * R::VP;
    if (c == NT) {
        for (int j = 0; j < D; j++) { xbptx::mbar_init(&full[j], 1); xbptx::mbar_init(&empty[j], W); xbptx::mbar_init(&cand[j], W); }
        xbptx::fence_barrier_init();
    }
    if (c < NT) {
        am[c] = c < C ? 1.0f : 0.0f;
        if (lane == 0) redm[w] = 1.0f;
    }
    __syncthreads();
    if (w == W) {                            // ---------------- service warp: copies ahead, labels behind
        if (lane == 0) {
            const float *abase = alpha + (size_t)n * R::VP, *bbase = beta + (size_t)n * R::VP, *mbase = bmax + (size_t)n * R::VP;
            auto fetch = [&](int t) {
                const int slot = t % D;
                const size_t rid = (size_t)t * N + n;
                R::fetch_row(ring + slot * R::ROWF, scores, rid, total_rows, &full[slot], 3 * R::VECB);
                bulk_g2s(xbptx::smem_u32(ringA + slot * R::VP), abase + (size_t)t * vrow, R::VECB, &full[slot]);
                bulk_g2s(xbptx::smem_u32(ringB + slot * R::VP), bbase + (size_t)(t + 1) * vrow, R::VECB, &full[slot]);
                bulk_g2s(xbptx::smem_u32(ringM + slot * R::VP), mbase + (size_t)(t + 1) * vrow, R::VECB, &full[slot]);
            };
            for (int j = 0; j < D - 1 && j < T; j++) fetch(j);
            for (int t = 0; t < T; t++) {
                if (t + D - 1 < T) {
                    if (t > 0) service_wait(&empty[(t - 1) % D], ((t - 1) / D) & 1);
                    fetch(t + D - 1);
                }
                // label of step t: first flat edge index among the per-warp maxima
                const int q = t % D;
                service_wait(&cand[q], (t / D) & 1);
                float bv = bval[q * W];
                int bi = bidx[q * W];
#pragma unroll
                for (int j = 1; j < W; j++) {
                    const float v = bval[q * W + j];
                    const int ix = bidx[q * W + j];
                    if (v > bv || (v == bv && ix < bi)) { bv = v; bi = ix; }
                }
                lab[t] = (int8_t)(bi % NZ);
            }
        }
    } else {
        const bool act = c < C;
        int src[NZ];
        src[0] = act ? c : 0;
#pragma unroll
        for (int k = 1; k < NZ; k++) src[k] = act ? (k - 1) * L::NP + c / NB : 0;
        const size_t prow = (size_t)N * S;
        float *prow_out = POST ? post_out + (size_t)n * S : nullptr;      // row t - 1 of this sequence
        for (int t = 0; t < T; t++) {
            const int slot = t % D;
            xbptx::mbar_wait(&full[slot], (t / D) & 1);
            compute_bar(NT);
            if (PSTAGE && t > 0) {
                const float *srow = pst + ((t - 1) & 1) * S;
                for (int i = c; i < S; i += NT) prow_out[i] = srow[i];
                prow_out += prow;
            }
            float *pout = !POST ? nullptr : PSTAGE ? pst + (t & 1) * S + c * NZ : post_out + ((size_t)t * N + n) * S + c * NZ;
            const float sc = xb_pow2_scale(red_max<W>(redm + (t & 1) * W));
            const float inv = XB_RCP(ringB[slot * R::VP + NT]);
            const float *M = ring + slot * R::ROWF + R::phase((size_t)t * N + n) + c * NZ;
            const float *A = ringA + slot * R::VP;
            const float *ac = am + (t & 1) * NT;
            float best = 0.0f, m = 0.0f;
            int besti = 0x7fffffff;
            float ev[NZ], av[NZ], bc = 0.0f, mc = 0.0f;
            if (act) {                        // everything this step needs from the ring slot, then release it
#pragma unroll
                for (int k = 0; k < NZ; k++) { ev[k] = edge_E<LIN>(M[k]); av[k] = A[src[k]]; }
                bc = ringB[slot * R::VP + c];
                mc = ringM[slot * R::VP + c];
            }
            __syncwarp();
            if (lane == 0) xbptx::mbar_arrive(&empty[slot]);
            if (act) {
#pragma unroll
                for (int k = 0; k < NZ; k++) {
                    const float we = XB_MUL(ev[k], bc);
                    const float p = XB_MUL(XB_MUL(av[k], we), inv);
                    if (POST) pout[k] = p;
                    const float v = XB_MUL(XB_ADD(p, XB_POST_EPS), XB_MUL(ac[src[k]], sc));
                    m = (k == 0) ? v : fmaxf(m, v);
                    const float cnd = XB_MUL(v, mc);
                    if (k == 0 || cnd > best) { best = cnd; besti = c * NZ + k; }
                }
                am[((t + 1) & 1) * NT + c] = m;
            }
            const float wm = warp_max_pos(m);
            if (lane == 0) redm[((t + 1) & 1) * W + w] = wm;
            // warp arg-max with first-index ties: candidates are non-negative, so their bit patterns order like the values
            const uint32_t key = act ? __float_as_uint(best) + 1u : 0u;      // + 1: an inactive lane never ties an active zero
            const uint32_t kmax = __reduce_max_sync(0xffffffffu, key);
            const int src_lane = __ffs(__ballot_sync(0xffffffffu, act && key == kmax)) - 1;
            if (src_lane >= 0) {
                best = __shfl_sync(0xffffffffu, best, src_lane);
                besti = __shfl_sync(0xffffffffu, besti, src_lane);
            }
            if (lane == 0) {
                bval[slot * W + w] = best;
                bidx[slot * W + w] = besti;
                xbptx::mbar_arrive(&cand[slot]);
            }
        }
    }
    __syncthreads();
    if (PSTAGE && T > 0 && c < NT) {                             // the last staged row
        const float *srow = pst + ((T - 1) & 1) * S;
        float *dst = post_out + ((size_t)(T - 1) * N + n) * S;
        for (int i = c; i < S; i += NT) dst[i] = srow[i];
    }
    pack_labels<NTT>(lab, scan, T, n, labels_out, seq_out, qs_out, lens_out, abc);
}

template <bool LIN, int NB, int SL>
int lin_impl(Lat<NB, SL>, xb_handle *h, const float *scores, int T, int N, int8_t *labels, int8_t *seq, int8_t *qs,
             int32_t *lens, float *post, cudaStream_t s) {
    using L = Lat<NB, SL>;
    using R = Ring<NB, SL>;
    constexpr int NTT = L::NT + 32;
    XB_REQUIRE(h, (reinterpret_cast<uintptr_t>(scores) & 15) == 0, "scores must be 16-byte aligned");
    // state vectors with pitch VP in handle workspace (xb_create sizes the three buffers for it)
    float *alpha = h->alpha, *beta = h->beta, *bmax = h->bmax;
    {
        xb_stage_timer tm(h, XB_ST_CRF_ALPHA, s);
        auto k = crf_lin_alpha_kernel<NB, SL, LIN>;
        const size_t sm = sizeof(float) * (L::D * R::ROWF + 2 * L::NT + 2 * L::W + 2) + 16 * L::D;
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, NTT, sm, s>>>(scores, T, N, alpha);
        XB_LAUNCH_CHECK(h);
    }
    {
        xb_stage_timer tm(h, XB_ST_CRF_BACKWARD, s);
        auto k = crf_lin_backward_kernel<NB, SL, LIN>;
        const size_t sm = sizeof(float) * (L::D * R::ROWF + L::D * R::VP + 4 * L::NT + 6 * L::W + 2) + 16 * L::D;
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, NTT, sm, s>>>(scores, alpha, T, N, beta, bmax);
        XB_LAUNCH_CHECK(h);
    }
    xb_stage_timer tm(h, XB_ST_CRF_VITERBI, s);
    const size_t sm = sizeof(float) * (L::D * R::ROWF + 3 * L::D * R::VP + 2 * L::NT + 2 * L::W + 2 * L::D * L::W + 2 + NTT + 1) +
                      24 * L::D + ((T + 15) / 16) * 16;
    Alphabet abc;
    for (int i = 0; i < 16; i++) abc.ch[i] = h->alphabet[i];
    if (post) {
        auto k = crf_lin_viterbi_kernel<NB, SL, LIN, true>;
        const size_t smp = sm + (L::S >= 1024 ? 2 * sizeof(float) * L::S : 0);        // + two staged posterior rows (see PSTAGE)
        if (int rc = xb_smem_attr(h, k, smp)) return rc;
        k<<<N, NTT, smp, s>>>(scores, alpha, beta, bmax, T, N, labels, seq, qs, lens, post, abc);
    } else {
        auto k = crf_lin_viterbi_kernel<NB, SL, LIN, false>;
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, NTT, sm, s>>>(scores, alpha, beta, bmax, T, N, labels, seq, qs, lens, nullptr, abc);
    }
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

}  // namespace

// Decode of (T, N, C*NZ) scores: labels / left-packed letters / lengths and, optionally, the posteriors.
// lin_input: the buffer holds E = exp(scores) (the fused head's output) instead of the scores.
int xb_decode_lin(xb_handle *h, const float *scores, int lin_input, int T, int N, int8_t *labels, int8_t *seq, int8_t *qs,
                  int32_t *lens, float *post, cudaStream_t s) {
    return lattice_dispatch(h, [&](auto lat) {
        return lin_input ? lin_impl<true>(lat, h, scores, T, N, labels, seq, qs, lens, post, s)
                         : lin_impl<false>(lat, h, scores, T, N, labels, seq, qs, lens, post, s);
    });
}
