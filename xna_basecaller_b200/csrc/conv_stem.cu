// Front of the convolution stem: Convolution(1->4,k5,p2)+swish, Convolution(4->16,k5,p2)+swish fused in one
// kernel (bonito/nn.py:57-68; built at bonito/crf/model.py:138-139,148-149), with the result emitted directly as
// the im2col rows of the third convolution (16->768, k19, stride 5, pad 9), so that conv3 runs as a tcgen05
// GEMM (gemm_tc.cu, EPI_CONV3).  The (N,4,L) and (N,16,L) intermediates of the reference never touch HBM.
//
// Row (chunk b, step t) of the im2col matrix holds c2[b, 5t-9+tap, ch] at column tap*16+ch for tap < 19, zero
// padded to 320 columns.  Padding semantics follow torch Conv1d: each layer sees zeros outside [0, L).
//
// One CTA = one chunk x 32 output steps: stages the 182 input samples it needs (halo included) in shared
// memory with coalesced loads, computes 178 conv1 and 174 conv2 positions in fp32, keeps conv2 in 16-bit
// channel-last form in shared memory, and writes the 32 overlapping 640-byte rows with 16-byte stores.
//
// DROP (the training forward and backward with dropout sites 0 / 1 active, xb_dropout.cuh): the fp32 conv1 values are
// masked before conv2 reads them and the conv2 values before they are rounded into the rows.  The mask is a function of
// the element index alone, so the halo positions a CTA shares with its neighbours get the same bits in both CTAs.
#include "xb_common.cuh"
#include "xb_dropout.cuh"

namespace {

constexpr int TT = 32;                         // output steps per CTA
constexpr int NP2 = 5 * TT + 14;               // conv2 positions needed: 5*t0-9 .. 5*(t0+TT-1)+9
constexpr int NP1 = NP2 + 4;
constexpr int NPX = NP1 + 4;
constexpr int THREADS = 256;

__device__ __forceinline__ float swishf(float x) { return x * __fdividef(1.0f, 1.0f + __expf(-x)); }

template <typename SIG> __device__ __forceinline__ float load_sig(const SIG *p, size_t i);
template <> __device__ __forceinline__ float load_sig<float>(const float *p, size_t i) { return __ldg(p + i); }
template <> __device__ __forceinline__ float load_sig<__half>(const __half *p, size_t i) { return __half2float(p[i]); }
template <> __device__ __forceinline__ float load_sig<int16_t>(const int16_t *p, size_t i) { return (float)p[i]; }

template <bool BF16, bool DROP, typename SIG>
__global__ void __launch_bounds__(THREADS)
conv12_im2col_kernel(const SIG *__restrict__ signal, int L, int T, const float *__restrict__ w1,
                     const float *__restrict__ b1, const float *__restrict__ w2, const float *__restrict__ b2,
                     uint16_t *__restrict__ rows, const xb_dropout drop) {
    using X = xb16<BF16>;
    __shared__ float sx[NPX];
    __shared__ float s1[NP1][4];
    __shared__ __align__(16) uint16_t s2[NP2 + 1][16];      // +1: the 16 zero pad columns of the last row read past tap 18
    __shared__ float sw1[20], sb1[4], sw2[320], sb2[16];

    const int b = blockIdx.y, t0 = blockIdx.x * TT, tid = threadIdx.x;
    const int p2_0 = 5 * t0 - 9;               // first conv2 position
    const int p1_0 = p2_0 - 2, px_0 = p1_0 - 2;
    const SIG *sig = signal + (size_t)b * L;

    for (int i = tid; i < 20; i += THREADS) sw1[i] = w1[i];
    for (int i = tid; i < 4; i += THREADS) sb1[i] = b1[i];
    for (int i = tid; i < 320; i += THREADS) sw2[i] = w2[i];
    for (int i = tid; i < 16; i += THREADS) sb2[i] = b2[i];
    for (int i = tid; i < NPX; i += THREADS) {
        int p = px_0 + i;
        sx[i] = (p >= 0 && p < L) ? load_sig<SIG>(sig, p) : 0.0f;
    }
    __syncthreads();
    for (int i = tid; i < NP1 * 4; i += THREADS) {
        int pos = i >> 2, ch = i & 3, p = p1_0 + pos;
        float v = 0.0f;
        if (p >= 0 && p < L) {
            v = sb1[ch];
#pragma unroll
            for (int k = 0; k < 5; k++) v = fmaf(sw1[ch * 5 + k], sx[pos + k], v);
            v = swishf(v);
            if (DROP && drop.on(0)) v = xb_dropout_apply(drop, 0, ((uint64_t)b * 4 + ch) * L + p, v);
        }
        s1[pos][ch] = v;
    }
    __syncthreads();
    for (int i = tid; i < (NP2 + 1) * 16; i += THREADS) {
        int pos = i >> 4, ch = i & 15, p = p2_0 + pos;
        float v = 0.0f;
        if (pos < NP2 && p >= 0 && p < L) {
            v = sb2[ch];
#pragma unroll
            for (int ci = 0; ci < 4; ci++)
#pragma unroll
                for (int k = 0; k < 5; k++) v = fmaf(sw2[(ch * 4 + ci) * 5 + k], s1[pos + k][ci], v);
            v = swishf(v);
            if (DROP && drop.on(1)) v = xb_dropout_apply(drop, 1, ((uint64_t)b * 16 + ch) * L + p, v);
        }
        typename X::T hv = X::from(v);
        s2[pos][ch] = *reinterpret_cast<uint16_t *>(&hv);
    }
    __syncthreads();
    // 32 rows x 40 16-byte vectors; vector v of row r = s2 bytes [(5r)*32 + 16v, +16), zero for v >= 38
    const uint4 *s2v = reinterpret_cast<const uint4 *>(&s2[0][0]);
    for (int i = tid; i < TT * 40; i += THREADS) {
        int r = i / 40, v = i - r * 40, t = t0 + r;
        if (t >= T) continue;
        uint4 val = make_uint4(0, 0, 0, 0);
        if (v < 38) val = s2v[r * 10 + v];
        reinterpret_cast<uint4 *>(rows + ((size_t)b * T + t) * XB_CONV3_K)[v] = val;
    }
}

template <bool BF16, typename SIG>
int launch(xb_handle *h, const void *signal, int N, int L, const xb_dropout *drop, cudaStream_t s) {
    const int T = L / XB_STRIDE;
    dim3 grid((T + TT - 1) / TT, N);
    const SIG *sig = reinterpret_cast<const SIG *>(signal);
    uint16_t *rows = reinterpret_cast<uint16_t *>(h->c2);
    if (drop && (drop->on(0) || drop->on(1)))
        conv12_im2col_kernel<BF16, true, SIG><<<grid, THREADS, 0, s>>>(sig, L, T, h->conv1_w, h->conv1_b, h->conv2_w,
                                                                      h->conv2_b, rows, *drop);
    else
        conv12_im2col_kernel<BF16, false, SIG><<<grid, THREADS, 0, s>>>(sig, L, T, h->conv1_w, h->conv1_b, h->conv2_w,
                                                                       h->conv2_b, rows, xb_dropout());
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

}  // namespace

// signal (N, L) -> h->c2 = im2col rows (N*T, 320) 16-bit; drop (may be NULL): the masks of dropout sites 0 and 1
int xb_conv12_im2col(xb_handle *h, const void *signal, int sig_dtype, int N, int L, cudaStream_t s, const xb_dropout *drop) {
    switch (sig_dtype) {        // activations are fp16 in both weight modes
        case XB_SIG_F32: return launch<false, float>(h, signal, N, L, drop, s);
        case XB_SIG_F16: return launch<false, __half>(h, signal, N, L, drop, s);
        case XB_SIG_I16: return launch<false, int16_t>(h, signal, N, L, drop, s);
    }
    return xb_fail(h, XB_ERR_ARG, "unknown signal dtype %d", sig_dtype);
}
