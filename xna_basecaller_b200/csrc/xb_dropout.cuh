// Dropout mask of the training step (rnn_encoder's drop_rate_bottom, crf/model.py): one counter-based generator that the
// forward, the backward and the halo recomputation of the convolution stem all evaluate, so that no mask is ever stored.
//
// Contract (restated in numpy by oracle/dropout.py; DESIGN section 2):
//   generator  Philox4x32-10 (Random123), M0 = 0xD2511F53, M1 = 0xCD9E8D57, W0 = 0x9E3779B9, W1 = 0xBB67AE85
//   key        (seed & 0xffffffff, seed >> 32)
//   counter    (e >> 2 low 32 bits, e >> 2 high 32 bits, site, 0); word e & 3 of the output decides element e
//   keep       word >= thr(p), thr(p) = min(floor(p * 2^32), 2^32 - 1) computed on the host in double from the float p
//   value      kept: x * scale, scale = (float)(1.0 / (1.0 - p)), multiplied in fp32 and rounded to the storage type;
//              dropped: 0
// Sites, in the order the reference applies them, and the element index e of each:
//   0  conv1 output (N, 4, L)       e = (n*4 + c)*L + l
//   1  conv2 output (N, 16, L)      e = (n*16 + c)*L + l
//   2  conv3 output (T, N, 768)     e = (t*N + n)*768 + f
//   3..6  output of LSTM layer site-3, (T, N, 768), t the forward time index whatever the layer's direction; e as for 2
#pragma once

#include "xb_common.cuh"

struct xb_dropout {
    uint32_t key[2] = {0, 0};
    uint32_t thr[XB_DROPOUT_SITES] = {};
    float scale[XB_DROPOUT_SITES] = {};
    uint32_t active = 0;         // bit s: p_s > 0.  A site whose bit is clear launches nothing and costs nothing
    __host__ __device__ bool on(int site) const { return (active >> site) & 1u; }
};

// p: host array of XB_DROPOUT_SITES probabilities (NULL: no dropout).  XB_ERR_ARG unless 0 <= p < 1 for every site.
inline int xb_dropout_init(xb_handle *h, xb_dropout *d, const float *p, uint64_t seed) {
    *d = xb_dropout();
    d->key[0] = (uint32_t)(seed & 0xffffffffu);
    d->key[1] = (uint32_t)(seed >> 32);
    for (int s = 0; s < XB_DROPOUT_SITES; s++) {
        const double ps = p ? (double)p[s] : 0.0;
        if (!(ps >= 0.0 && ps < 1.0)) return xb_fail(h, XB_ERR_ARG, "dropout probability of site %d must lie in [0, 1) (got %g)", s, ps);
        const double t = ps * 4294967296.0;
        d->thr[s] = t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
        d->scale[s] = (float)(1.0 / (1.0 - ps));
        if (ps > 0.0) d->active |= 1u << s;
    }
    return XB_OK;
}

__device__ __forceinline__ uint4 xb_philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    }
    return c;
}

// the four words that decide elements 4q .. 4q + 3 of a site
__device__ __forceinline__ uint4 xb_dropout_words(const xb_dropout &d, int site, uint64_t q) {
    return xb_philox4x32_10(make_uint4((uint32_t)q, (uint32_t)(q >> 32), (uint32_t)site, 0u), d.key[0], d.key[1]);
}

__device__ __forceinline__ bool xb_dropout_keep(const xb_dropout &d, int site, uint64_t e) {
    const uint4 w = xb_dropout_words(d, site, e >> 2);
    const uint32_t j = (uint32_t)e & 3u;
    const uint32_t word = j == 0 ? w.x : j == 1 ? w.y : j == 2 ? w.z : w.w;
    return word >= d.thr[site];
}

// x times the mask of element e (fp32 values: the convolution stem)
__device__ __forceinline__ float xb_dropout_apply(const xb_dropout &d, int site, uint64_t e, float x) {
    return xb_dropout_keep(d, site, e) ? x * d.scale[site] : 0.0f;
}

// Eight 16-bit values (fp16, or bf16 with BF16) of elements e .. e + 7, e a multiple of 8: two generator calls
template <bool BF16>
__device__ __forceinline__ uint4 xb_dropout8(const xb_dropout &d, int site, uint64_t e, uint4 v) {
    const uint4 a = xb_dropout_words(d, site, e >> 2), b = xb_dropout_words(d, site, (e >> 2) + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t u[4] = {v.x, v.y, v.z, v.w};
    const uint32_t thr = d.thr[site];
    const float sc = d.scale[site];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        float2 f = xb16<BF16>::unpack(u[j]);
        f.x = w[2 * j] >= thr ? f.x * sc : 0.0f;
        f.y = w[2 * j + 1] >= thr ? f.y * sc : 0.0f;
        u[j] = xb16<BF16>::pack(f.x, f.y);
    }
    return make_uint4(u[0], u[1], u[2], u[3]);
}
