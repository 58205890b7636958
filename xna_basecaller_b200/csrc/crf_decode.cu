// CTC-CRF scans on RAW scores for sm_100a, in the log domain: Log-semiring forward (alpha / logZ), backward scans in
// either semiring, Max-semiring forward sweep with arg-max edges and labels (CTC_CRF.logZ / forward_scores /
// backward_scores / viterbi).  decode_batch (posteriors + max-marginal Viterbi) lives in crf_decode_lin.cu.
//
// Reference semantics: bonito/crf/model.py:26-46 (idx, logZ), :51-61 (forward/backward scores), :92-100
// (viterbi, path_to_str), :215-218 (decode_batch); bonito/crf/basecall.py:56-76 (left-packed rows); the
// seqdist semiring algebra as restated in oracle/seqdist_restated.py.  The arithmetic contract (operation
// order, reduction tree, exp/log) is the one written at the top of oracle/c/crf_exact.c; the two must stay
// in lock step because the tests demand bit-equal labels.
//
// Mapping: one CTA per sequence, one thread per CRF state (C = n_base^state_len; 128 threads for the
// 5-letter alphabet, 224 for 6 letters), so all N sequences are resident at once (N/148 CTAs per SM) and
// the serial dependence over T is hidden by the other CTAs of the SM.  The score rows of a sequence are
// streamed through a cp.async ring in shared memory several steps ahead of the recurrence (HBM-bound
// part); state vectors ping-pong in shared memory with one barrier per step.
#include "xb_common.cuh"
#include "xb_exact_math.h"
#include "crf_lattice.cuh"

using namespace xbcrf;

namespace {

// --------------------------------------------------------------------------------------------------
// Forward sweep, Log or Max semiring: alpha (T+1,N,C) and / or logZ (N).      grid = N, block = NT
template <int NB, int SL, bool USE_MAX>
__global__ void __launch_bounds__(Lat<NB, SL>::NT)
crf_alpha_kernel(const float *__restrict__ scores, int T, int N, float *__restrict__ alpha_out,
                 float *__restrict__ logz_out) {
    using L = Lat<NB, SL>;
    constexpr int C = L::C, NZ = L::NZ, S = L::S, NT = L::NT, W = L::W, D = L::D;
    extern __shared__ __align__(16) float smem[];
    float *ring = smem;              // D * S
    float *a = ring + D * S;         // 2 * NT
    float *red = a + 2 * NT;         // 2 * W
    const int n = blockIdx.x, c = threadIdx.x, lane = c & 31, w = c >> 5;
    const bool act = c < C;
    const float *base = scores + (size_t)n * S;
    const size_t row = (size_t)N * S;

#pragma unroll
    for (int j = 0; j < D - 1; j++) {
        if (j < T) copy_row<S, NT>(ring + j * S, base + (size_t)j * row);
        cp_async_commit();
    }
    a[c] = 0.0f;
    if (alpha_out && act) alpha_out[(size_t)n * C + c] = 0.0f;
    int src[NZ];
    src[0] = act ? c : 0;
#pragma unroll
    for (int k = 1; k < NZ; k++) src[k] = act ? (k - 1) * L::NP + c / NB : 0;

    // running pointers instead of per-step 64-bit index arithmetic: next row to fetch, next alpha row to write
    const float *fetch = base + (size_t)(D - 1) * row;
    float *aout = alpha_out ? alpha_out + ((size_t)N + n) * C + c : nullptr;
    const size_t arow = (size_t)N * C;
    for (int t = 0; t < T; t++) {
        cp_async_wait<D - 2>();
        __syncthreads();
        {
            int r = t + D - 1;
            if (r < T) copy_row<S, NT>(ring + (r % D) * S, fetch);
            fetch += row;
            cp_async_commit();
        }
        const float *M = ring + (t % D) * S + c * NZ;
        const float *ac = a + (t & 1) * NT;
        float *an = a + ((t + 1) & 1) * NT;
        if (act) {
            float x[NZ], m;
#pragma unroll
            for (int k = 0; k < NZ; k++) {
                x[k] = XB_ADD(M[k], ac[src[k]]);
                m = (k == 0) ? x[k] : fmaxf(m, x[k]);
            }
            float v = USE_MAX ? m : lse_exact<NZ>(x, m);
            an[c] = v;
            if (aout) *aout = v;
        }
        if (aout) aout += arow;
    }
    __syncthreads();
    if (logz_out) {
        float v = act ? a[(T & 1) * NT + c] : -INFINITY;
        float m = warp_max(v);
        if (lane == 0) red[w] = m;
        __syncthreads();
        m = red[0];
#pragma unroll
        for (int i = 1; i < W; i++) m = fmaxf(m, red[i]);
        float e = act ? xb_expf(XB_SUB(v, m)) : 0.0f;
        e = warp_sum_tree(e);
        if (lane == 0) red[W + w] = e;
        __syncthreads();
        if (c == 0) {
            float s = red[W];
            for (int i = 1; i < W; i++) s = XB_ADD(s, red[W + i]);
            logz_out[n] = USE_MAX ? m : XB_ADD(m, xb_logf(s));        // Max semiring: the best path's score
        }
    }
}

// --------------------------------------------------------------------------------------------------
// Plain backward scan over the raw scores in either semiring: out (T+1,N,C).  Used for
// CTC_CRF.backward_scores (Log) and for the Max-beta of CTC_CRF.viterbi on arbitrary scores.
template <int NB, int SL, bool USE_MAX>
__global__ void __launch_bounds__(Lat<NB, SL>::NT)
crf_bscan_kernel(const float *__restrict__ scores, int T, int N, float *__restrict__ out) {
    using L = Lat<NB, SL>;
    constexpr int C = L::C, NZ = L::NZ, S = L::S, NT = L::NT, D = L::D;
    extern __shared__ __align__(16) float smem[];
    float *ring = smem;
    float *b = ring + D * S;         // 2 * NT
    const int n = blockIdx.x, c = threadIdx.x;
    const bool act = c < C;
    const float *base = scores + (size_t)n * S;
    const size_t row = (size_t)N * S;
#pragma unroll
    for (int j = 0; j < D - 1; j++) {
        if (j < T) copy_row<S, NT>(ring + j * S, base + (size_t)(T - 1 - j) * row);
        cp_async_commit();
    }
    b[c] = 0.0f;
    if (act) out[((size_t)T * N + n) * C + c] = 0.0f;
    const int kk = act ? 1 + c / L::NP : 1, cb = act ? (c % L::NP) * NB : 0;
    for (int i = 0; i < T; i++) {
        const int t = T - 1 - i;
        cp_async_wait<D - 2>();
        __syncthreads();
        {
            int r = i + D - 1;
            if (r < T) copy_row<S, NT>(ring + (r % D) * S, base + (size_t)(T - 1 - r) * row);
            cp_async_commit();
        }
        const float *M = ring + (i % D) * S;
        const float *b1 = b + (i & 1) * NT;
        float *b0 = b + ((i + 1) & 1) * NT;
        if (act) {
            float y[NZ], m;
            y[0] = XB_ADD(M[c * NZ], b1[c]);
            m = y[0];
#pragma unroll
            for (int j = 0; j < NB; j++) {
                y[1 + j] = XB_ADD(M[(cb + j) * NZ + kk], b1[cb + j]);
                m = fmaxf(m, y[1 + j]);
            }
            float v = USE_MAX ? m : lse_exact<NZ>(y, m);
            b0[c] = v;
            out[((size_t)t * N + n) * C + c] = v;
        }
    }
}

// --------------------------------------------------------------------------------------------------
// Forward sweep, Max semiring, over the scores with the stored Max-beta: arg-max edge per step -> edges_out and / or
// its label (edge % NZ) -> labels_out.
template <int NB, int SL>
__global__ void __launch_bounds__(Lat<NB, SL>::NT)
crf_viterbi_fwd_kernel(const float *__restrict__ scores, const float *__restrict__ bmax, int T, int N,
                       int8_t *__restrict__ labels_out, int32_t *__restrict__ edges_out) {
    using L = Lat<NB, SL>;
    constexpr int C = L::C, NZ = L::NZ, S = L::S, NT = L::NT, W = L::W, D = L::D;
    extern __shared__ __align__(16) float smem[];
    float *ring = smem;                  // D * S
    float *ringB = ring + D * S;         // D * NT
    float *am = ringB + D * NT;          // 2 * NT
    float *bval = am + 2 * NT;           // 2 * W
    int *bidx = reinterpret_cast<int *>(bval + 2 * W);      // 2 * W
    const int n = blockIdx.x, c = threadIdx.x, lane = c & 31, w = c >> 5;
    const bool act = c < C;
    const float *base = scores + (size_t)n * S;
    const size_t row = (size_t)N * S;
    const float *bbase = bmax + (size_t)n * C;
    const size_t brow = (size_t)N * C;
    // thread 0: step t's arg-max over the per-warp candidates (first index on ties)
    auto finish = [&](int t) {
        const int q = t & 1;
        float bv = bval[q * W];
        int bi = bidx[q * W];
        for (int j = 1; j < W; j++) {
            float v = bval[q * W + j];
            int ix = bidx[q * W + j];
            if (v > bv || (v == bv && ix < bi)) { bv = v; bi = ix; }
        }
        if (labels_out) labels_out[(size_t)n * T + t] = (int8_t)(bi % NZ);
        if (edges_out) edges_out[(size_t)n * T + t] = bi;
    };

#pragma unroll
    for (int j = 0; j < D - 1; j++) {
        if (j < T) {
            copy_row<S, NT>(ring + j * S, base + (size_t)j * row);
            if (act) cp_async4(ringB + j * NT + c, bbase + (size_t)(j + 1) * brow + c);
        }
        cp_async_commit();
    }
    am[c] = 0.0f;
    int src[NZ];
    src[0] = act ? c : 0;
#pragma unroll
    for (int k = 1; k < NZ; k++) src[k] = act ? (k - 1) * L::NP + c / NB : 0;

    const float *fetchM = base + (size_t)(D - 1) * row;          // running pointers: row r = t + D - 1, Max-beta row r + 1
    const float *fetchB = bbase + (size_t)D * brow + c;
    for (int t = 0; t < T; t++) {
        cp_async_wait<D - 2>();
        __syncthreads();
        {
            int r = t + D - 1;
            if (r < T) {
                copy_row<S, NT>(ring + (r % D) * S, fetchM);
                if (act) cp_async4(ringB + (r % D) * NT + c, fetchB);
            }
            fetchM += row;
            fetchB += brow;
            cp_async_commit();
        }
        if (c == 0 && t > 0) finish(t - 1);
        const float *M = ring + (t % D) * S + c * NZ;
        const float *ac = am + (t & 1) * NT;
        float *an = am + ((t + 1) & 1) * NT;
        float best = -INFINITY;
        int besti = 0x7fffffff;
        if (act) {
            const float bc = ringB[(t % D) * NT + c];
            float m;
#pragma unroll
            for (int k = 0; k < NZ; k++) {
                float v = XB_ADD(M[k], ac[src[k]]);
                m = (k == 0) ? v : fmaxf(m, v);
                float sc = XB_ADD(v, bc);
                if (k == 0 || sc > best) { best = sc; besti = c * NZ + k; }
            }
            an[c] = m;
        }
        // warp arg-max with first-index ties: one integer REDUX on an order-preserving key, then the lowest lane that
        // holds the maximum (lanes are ordered by state, and each lane already kept its lowest edge index)
        {
            const uint32_t bits = __float_as_uint(best + 0.0f);                 // + 0.0f: -0 and +0 get the same key
            const uint32_t key = act ? (bits ^ ((bits >> 31) ? 0xffffffffu : 0x80000000u)) : 0u;
            const uint32_t kmax = __reduce_max_sync(0xffffffffu, key);
            const int src_lane = __ffs(__ballot_sync(0xffffffffu, act && key == kmax)) - 1;
            if (src_lane >= 0) {
                best = __shfl_sync(0xffffffffu, best, src_lane);
                besti = __shfl_sync(0xffffffffu, besti, src_lane);
            }
        }
        if (lane == 0) { bval[(t & 1) * W + w] = best; bidx[(t & 1) * W + w] = besti; }
    }
    __syncthreads();
    if (c == 0 && T > 0) finish(T - 1);
}

template <int NB, int SL> size_t smem_alpha() {
    using L = Lat<NB, SL>;
    return sizeof(float) * (L::D * L::S + 2 * L::NT + 2 * L::W);
}
template <int NB, int SL> size_t smem_bscan() {
    using L = Lat<NB, SL>;
    return sizeof(float) * (L::D * L::S + 2 * L::NT);
}
template <int NB, int SL> size_t smem_vit() {
    using L = Lat<NB, SL>;
    return sizeof(float) * (L::D * L::S + L::D * L::NT + 2 * L::NT + 4 * L::W);
}

template <int NB, int SL>
int alpha_impl(Lat<NB, SL>, xb_handle *h, const float *scores, int T, int N, float *alpha, float *logz, int use_max,
               cudaStream_t s) {
    using L = Lat<NB, SL>;
    size_t sm = smem_alpha<NB, SL>();
    if (use_max) {
        auto k = crf_alpha_kernel<NB, SL, true>;
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, L::NT, sm, s>>>(scores, T, N, alpha, logz);
    } else {
        auto k = crf_alpha_kernel<NB, SL, false>;
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, L::NT, sm, s>>>(scores, T, N, alpha, logz);
    }
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
template <int NB, int SL>
int backward_impl(Lat<NB, SL>, xb_handle *h, const float *scores, int T, int N, float *bmax, float *beta, int mode,
                  cudaStream_t s) {
    using L = Lat<NB, SL>;
    if (mode == 1) {
        auto k = crf_bscan_kernel<NB, SL, true>;
        size_t sm = smem_bscan<NB, SL>();
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, L::NT, sm, s>>>(scores, T, N, bmax);
    } else {
        auto k = crf_bscan_kernel<NB, SL, false>;
        size_t sm = smem_bscan<NB, SL>();
        if (int rc = xb_smem_attr(h, k, sm)) return rc;
        k<<<N, L::NT, sm, s>>>(scores, T, N, beta);
    }
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
template <int NB, int SL>
int vit_impl(Lat<NB, SL>, xb_handle *h, const float *scores, const float *bmax, int T, int N, int8_t *labels, int32_t *edges,
             cudaStream_t s) {
    using L = Lat<NB, SL>;
    auto k = crf_viterbi_fwd_kernel<NB, SL>;
    size_t sm = smem_vit<NB, SL>();
    if (int rc = xb_smem_attr(h, k, sm)) return rc;
    k<<<N, L::NT, sm, s>>>(scores, bmax, T, N, labels, edges);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

}  // namespace

int xb_decode_alpha(xb_handle *h, const float *scores, int T, int N, float *alpha, float *logz, int use_max, cudaStream_t s) {
    xb_stage_timer tm(h, XB_ST_CRF_ALPHA, s);
    return lattice_dispatch(h, [&](auto lat) { return alpha_impl(lat, h, scores, T, N, alpha, logz, use_max, s); });
}

// mode 1: Max-semiring backward scan of the raw scores into bmax;  mode 2: Log-semiring scan into beta
int xb_decode_backward(xb_handle *h, const float *scores, int T, int N, float *bmax, float *beta, int mode, cudaStream_t s) {
    xb_stage_timer tm(h, XB_ST_CRF_BACKWARD, s);
    return lattice_dispatch(h, [&](auto lat) { return backward_impl(lat, h, scores, T, N, bmax, beta, mode, s); });
}

int xb_decode_viterbi_fwd(xb_handle *h, const float *scores, const float *bmax, int T, int N, int8_t *labels, int32_t *edges,
                          cudaStream_t s) {
    xb_stage_timer tm(h, XB_ST_CRF_VITERBI, s);
    return lattice_dispatch(h, [&](auto lat) { return vit_impl(lat, h, scores, bmax, T, N, labels, edges, s); });
}
