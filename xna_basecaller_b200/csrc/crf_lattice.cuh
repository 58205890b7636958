// Shared pieces of the CRF scan kernels (crf_decode.cu: Log / Max semiring scans on raw scores; crf_decode_lin.cu: the
// linear-domain decode): lattice constants, the list of supported lattices and the dispatch over it, the cp.async
// score-row ring, warp reductions with a fixed evaluation order.
#pragma once
#include "xb_common.cuh"
#include "xb_exact_math.h"

namespace xbcrf {

template <int NB, int SL> struct Lat {
    static constexpr int ipow(int b, int e) { return e == 0 ? 1 : b * ipow(b, e - 1); }
    static constexpr int C = ipow(NB, SL);
    static constexpr int NP = ipow(NB, SL - 1);
    static constexpr int NZ = NB + 1;
    static constexpr int S = C * NZ;                   // scores per (t, n)
    static constexpr int NT = ((C + 31) / 32) * 32;    // threads per CTA
    static constexpr int W = NT / 32;
    static constexpr int D0 = 24576 / (S * 4);
    static constexpr int D = D0 < 2 ? 2 : (D0 > 8 ? 8 : D0);   // ring depth (rows in flight + 1)
    static_assert(S % 2 == 0, "row must be a whole number of 8-byte chunks");
};

// The lattices (n_base, state_len) the CRF kernels are compiled for -- the one list of them: f(Lat<NB, SL>()) for one of
// these, unsupported() for any other.
template <typename F, typename U> int for_lattice(int n_base, int state_len, F &&f, U &&unsupported) {
    switch (n_base * 10 + state_len) {
        case 43: return f(Lat<4, 3>());
        case 53: return f(Lat<5, 3>());
        case 63: return f(Lat<6, 3>());
        case 44: return f(Lat<4, 4>());
        case 22: return f(Lat<2, 2>());
    }
    return unsupported();
}

inline bool lattice_supported(int n_base, int state_len) {
    return for_lattice(n_base, state_len, [](auto) { return 1; }, [] { return 0; });
}

// f(Lat<NB, SL>()) for the handle's lattice
template <typename F> int lattice_dispatch(xb_handle *h, F &&f) {
    return for_lattice(h->n_base, h->state_len, f, [h] {
        return xb_fail(h, XB_ERR_UNSUPPORTED, "no CRF kernel compiled for n_base=%d state_len=%d", h->n_base, h->state_len);
    });
}

__device__ __forceinline__ void cp_async4(float *dst, const float *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src));
}
__device__ __forceinline__ void cp_async8(float *dst, const float *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int NPEND> __device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(NPEND));
}

// One score row global -> shared in 8-byte cp.async pieces (rows are only 8-byte aligned: S * 4 = 3000 B for n_base 5).
// Fully unrolled on one shared and one global base address with immediate offsets: the rolled loop spent ~24 instructions
// per piece on address arithmetic -- a quarter of the alpha sweep's instruction count.
template <int NFLOATS, int NT> __device__ __forceinline__ void copy_row(float *dst, const float *src) {
    constexpr int NCOPY = NFLOATS / 2, ROUNDS = (NCOPY + NT - 1) / NT;
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst) + threadIdx.x * 8u;
    const char *g = reinterpret_cast<const char *>(src) + threadIdx.x * 8u;
#pragma unroll
    for (int k = 0; k < ROUNDS; k++)
        if ((k + 1) * NT <= NCOPY || k * NT + (int)threadIdx.x < NCOPY)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d + (uint32_t)(k * NT * 8)), "l"(g + k * NT * 8));
}

// warp maximum with one integer REDUX on an order-preserving key (max is exact, so any evaluation order gives the same
// value; +0.0f folds -0 into +0 so that the key order equals the float order)
__device__ __forceinline__ float warp_max(float v) {
    const uint32_t bits = __float_as_uint(v + 0.0f);
    const uint32_t key = bits ^ ((bits >> 31) ? 0xffffffffu : 0x80000000u);
    const uint32_t kmax = __reduce_max_sync(0xffffffffu, key);
    return __uint_as_float(kmax ^ ((kmax >> 31) ? 0x80000000u : 0xffffffffu));
}
// xor butterfly: every lane ends with the same bits (a+b == b+a), see oracle/c/crf_exact.c tree_sum()
__device__ __forceinline__ float warp_sum_tree(float v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = XB_ADD(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

template <int NZ> __device__ __forceinline__ float lse_exact(const float (&x)[NZ], float m) {
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < NZ; k++) {
        float e = xb_expf_le0(XB_SUB(x[k], m));
        s = (k == 0) ? e : XB_ADD(s, e);
    }
    return XB_ADD(m, xb_logf_norm(s));
}


struct Alphabet { char ch[16]; };

// Labels of one sequence (shared memory, T entries) -> labels_out row, left-packed letters (path_to_str,
// bonito/crf/model.py:97-100; bonito/crf/basecall.py:56-76), dummy quality 'O', length.  Whole CTA; scan = NT + 1 ints.
template <int NT>
__device__ __forceinline__ void pack_labels(const int8_t *lab, int *scan, int T, int n, int8_t *__restrict__ labels_out,
                                            int8_t *__restrict__ seq_out, int8_t *__restrict__ qs_out,
                                            int32_t *__restrict__ lens_out, const Alphabet &abc) {
    const int c = threadIdx.x;
    if (labels_out)
        for (int t = c; t < T; t += NT) labels_out[(size_t)n * T + t] = lab[t];
    if (!seq_out) return;
    const int per = (T + NT - 1) / NT;                     // thread c owns steps [c*per, (c+1)*per)
    const int lo = min(c * per, T), hi = min(lo + per, T);
    int cnt = 0;
    for (int t = lo; t < hi; t++) cnt += lab[t] != 0;
    scan[c + 1] = cnt;
    if (c == 0) scan[0] = 0;
    __syncthreads();
    if (c == 0)
        for (int j = 1; j <= NT; j++) scan[j] += scan[j - 1];
    __syncthreads();
    int pos = scan[c];
    const int total = scan[NT];
    for (int t = lo; t < hi; t++) {
        int l = lab[t];
        if (l != 0) {
            seq_out[(size_t)n * T + pos] = (int8_t)abc.ch[l];
            if (qs_out) qs_out[(size_t)n * T + pos] = (int8_t)'O';
            pos++;
        }
    }
    for (int p = total + c; p < T; p += NT) {
        seq_out[(size_t)n * T + p] = 0;
        if (qs_out) qs_out[(size_t)n * T + p] = 0;
    }
    if (c == 0 && lens_out) lens_out[n] = total;
}

}  // namespace xbcrf
