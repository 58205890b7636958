// C ABI of libxna_b200.so (include/xna_basecaller.h): handle life cycle, weight repacking, the encoder
// pipeline (conv stem -> 5 LSTM layers -> CRF head), the CRF decode entry points and the host-buffer call.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "xb_common.cuh"
#include "xb_gemm.cuh"

thread_local std::string xb_global_err;

int xb_fail(xb_handle *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    xb_global_err = buf;
    return code;
}

struct xb_dropout;
int xb_conv12_im2col(xb_handle *h, const void *signal, int sig_dtype, int N, int L, cudaStream_t s,
                     const xb_dropout *drop = nullptr);
int xb_lstm_recurrence_persistent(xb_handle *h, int layer, void *y_tnc, int T, int N, int reverse, cudaStream_t s, void *save = nullptr);
int xb_inproj_launch(xb_handle *h, const void *x, const void *w_ih, const float *bias, void *gates, int M, cudaStream_t s);
int xb_head_astationary_launch(xb_handle *h, const void *x, const void *w, int w_rows, const float *bias, int head_rows,
                               float *scores, int ldo, int M, int exp_out, cudaStream_t s);
int xb_preprocess_impl(xb_handle *h, const int16_t *raw, const int64_t *read_offset, const int32_t *read_len,
                       const double *scaling, const int32_t *offset, int n_reads, float *out, int32_t *out_len,
                       float *stats, cudaStream_t s);
int xb_ctc_loss_bwd_impl(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                         const int32_t *lengths, int normalise, const float *grad_loss, float *alpha_ws, float *grad,
                         cudaStream_t s);
int xb_ctc_loss_impl(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                     const int32_t *lengths, int normalise, float *loss, cudaStream_t s);
int xb_stitch_impl(xb_handle *h, const int8_t *rows, int T, const int32_t *chunk_first, const int32_t *chunk_count,
                   const int32_t *read_len, int n_reads, int chunksize, int overlap, int stride, int reverse, int8_t *out,
                   int out_stride, int32_t *out_len, cudaStream_t s);

void xb_train_free(xb_handle *h);
int xb_beam_search_impl(xb_handle *h, const float *scores, const float *beta, int T, int N, int beam_width, float beam_cut,
                        int8_t *seq, int8_t *qstring, int8_t *moves, int32_t *lens, cudaStream_t s);
int xb_onehot_edges(xb_handle *h, const int32_t *edges_nt, int T, int N, int S, float *post, cudaStream_t s);
int xb_gather_chunks_impl(xb_handle *h, const void *signal, int sig_dtype, const int64_t *read_offset,
                          const int32_t *read_len, const int32_t *chunk_read, const int32_t *chunk_start, int n_chunks,
                          int L, float *out, cudaStream_t s);

namespace {

int ipow(int b, int e) { int r = 1; while (e-- > 0) r *= b; return r; }

template <typename T> int dev_alloc(xb_handle *h, T **p, size_t count) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T));
    if (e != cudaSuccess)
        return xb_fail(h, XB_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
    *p = reinterpret_cast<T *>(q);
    return XB_OK;
}
int dev_alloc_bytes(xb_handle *h, void **p, size_t bytes) { return dev_alloc<uint8_t>(h, reinterpret_cast<uint8_t **>(p), bytes); }

// ---- weight repacking ------------------------------------------------------------------------------
// dst (rows_dst, cols_dst) 16-bit <- src fp32; mode 0: plain rows (zero padding past rows_src / cols_src);
// mode 1: LSTM gate interleave, dst row j*128 + g*32 + u <- src row g*768 + j*32 + u;
// mode 2: conv3 (768,16,19) -> (768, 320) with column tap*16 + ch;
// mode 3: LSTM unit-major interleave, dst row j*128 + u*4 + g <- src row g*768 + j*32 + u (the input projection
//         of the persistent kernel: the four gates of a unit are adjacent in a row of G);
// mode 4: W_hh of the persistent kernel: dst row j*128 + q*32 + g*8 + ul <- src row g*768 + j*32 + q*8 + ul: within a
//         TMEM lane quarter the rows are gate-major, which is what tcgen05.ld.16x256b hands to one thread.
template <bool BF16>
__global__ void repack_kernel(const float *__restrict__ src, uint16_t *__restrict__ dst, int rows_dst, int cols_dst,
                              int rows_src, int cols_src, int mode) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows_dst * cols_dst) return;
    int r = (int)(i / cols_dst), c = (int)(i % cols_dst);
    float v = 0.0f;
    if (mode == 0) {
        if (r < rows_src && c < cols_src) v = src[(size_t)r * cols_src + c];
    } else if (mode == 1) {
        int j = r >> 7, g = (r >> 5) & 3, u = r & 31;
        v = src[(size_t)(g * XB_FEATURES + j * 32 + u) * cols_src + c];
    } else if (mode == 3) {
        int j = r >> 7, u = (r >> 2) & 31, g = r & 3;
        v = src[(size_t)(g * XB_FEATURES + j * 32 + u) * cols_src + c];
    } else if (mode == 4) {
        int j = r >> 7, q = (r >> 5) & 3, g = (r >> 3) & 3, ul = r & 7;
        v = src[(size_t)(g * XB_FEATURES + j * 32 + q * 8 + ul) * cols_src + c];
    } else if (mode == 5 || mode == 6) {      // transposes for the training backward, stored as bf16: dst (cols_src.., rows_src..) = src^T
        if (mode == 5) { if (r < cols_src && c < rows_src) v = src[(size_t)c * cols_src + r]; }
        else {                                 // conv3 (768,16,19) -> (320, 768): row tap*16 + ch
            int tap = r >> 4, ch = r & 15;
            if (tap < XB_WINLEN) v = src[((size_t)c * XB_C2_CH + ch) * XB_WINLEN + tap];
        }
        __nv_bfloat16 bv = __float2bfloat16_rn(v);
        dst[i] = *reinterpret_cast<uint16_t *>(&bv);
        return;
    } else {
        int tap = c >> 4, ch = c & 15;
        if (tap < XB_WINLEN) v = src[((size_t)r * XB_C2_CH + ch) * XB_WINLEN + tap];
    }
    // Every kernel multiplies fp16 operands.  XB_FLAG_BF16 ("bf16 weights") rounds the weight to bfloat16 first -- the
    // value a bf16 checkpoint / bf16 autocast holds -- and stores that number as fp16: 8 mantissa bits fit into 11, so the
    // conversion is exact for every weight above the fp16 subnormal range (|w| >= 6e-5; below it the absolute error is
    // <= 3e-8).  tcgen05 kind::f16 does not accept an fp16 x bf16 operand pair (illegal instruction, measured), and
    // bf16 activations (h, the hoisted input projection) would cost 5x the score error (tests/precision_attribution.py).
    if (BF16) v = __bfloat162float(__float2bfloat16_rn(v));
    __half hv = __float2half_rn(v);
    dst[i] = *reinterpret_cast<uint16_t *>(&hv);
}
__global__ void lstm_bias_kernel(const float *__restrict__ b_ih, const float *__restrict__ b_hh, float *__restrict__ dst,
                                 int mode) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= XB_GATES) return;
    int j = r >> 7, g = (r >> 5) & 3, u = r & 31;
    if (mode == 3) { u = (r >> 2) & 31; g = r & 3; }
    int s = g * XB_FEATURES + j * 32 + u;
    dst[r] = b_ih[s] + b_hh[s];
}

int repack(xb_handle *h, const float *src, void *dst, int rows_dst, int cols_dst, int rows_src, int cols_src, int mode,
           cudaStream_t s) {
    size_t n = (size_t)rows_dst * cols_dst;
    int blocks = (int)((n + 255) / 256);
    if (h->bf16)
        repack_kernel<true><<<blocks, 256, 0, s>>>(src, reinterpret_cast<uint16_t *>(dst), rows_dst, cols_dst, rows_src, cols_src, mode);
    else
        repack_kernel<false><<<blocks, 256, 0, s>>>(src, reinterpret_cast<uint16_t *>(dst), rows_dst, cols_dst, rows_src, cols_src, mode);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

int check_tn(xb_handle *h, int T, int N) {
    XB_CUDA(h, cudaSetDevice(h->device));      // every compute entry point passes here: kernels go to the handle's device
    XB_REQUIRE(h, T > 0 && N > 0, "T and N must be positive (got T=%d N=%d)", T, N);
    XB_REQUIRE(h, T <= h->max_T && N <= h->max_N, "T=%d N=%d exceed the handle capacity max_T=%d max_N=%d", T, N, h->max_T,
               h->max_N);
    return XB_OK;
}

}  // namespace

extern "C" {

int xb_abi_version(void) { return XB_ABI_VERSION; }

const char *xb_last_error(const xb_handle *h) { return h ? h->err.c_str() : xb_global_err.c_str(); }

int64_t xb_launch_count(const xb_handle *h) { return h ? h->launches : 0; }

int xb_set_profiling(xb_handle *h, int on) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    h->profiling = on != 0;
    return XB_OK;
}

int xb_stage_times(xb_handle *h, float *ms, int *spans) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, ms && spans, "NULL buffer");
    for (int i = 0; i < XB_ST_COUNT; i++) { ms[i] = 0.f; spans[i] = 0; }
    for (auto &sp : h->spans) {
        XB_CUDA(h, cudaEventSynchronize(sp.b));
        float t = 0.f;
        XB_CUDA(h, cudaEventElapsedTime(&t, sp.a, sp.b));
        ms[sp.stage] += t;
        spans[sp.stage]++;
        h->event_pool.push_back(sp.a);
        h->event_pool.push_back(sp.b);
    }
    h->spans.clear();
    return XB_OK;
}

int xb_create(xb_handle **out, int device, int max_N, int max_T, int n_base, int state_len, const char *alphabet, int flags) {
    if (!out) return xb_fail(nullptr, XB_ERR_ARG, "xb_create: out is NULL");
    *out = nullptr;
    if (max_N <= 0 || max_T <= 0) return xb_fail(nullptr, XB_ERR_ARG, "xb_create: max_N and max_T must be positive");
    if (!alphabet || (int)strlen(alphabet) != n_base + 1 || n_base + 1 > 15)
        return xb_fail(nullptr, XB_ERR_ARG, "xb_create: alphabet must have n_base+1 letters (blank first)");
    int key = n_base * 10 + state_len;
    if (!(key == 43 || key == 53 || key == 63 || key == 44 || key == 22))
        return xb_fail(nullptr, XB_ERR_UNSUPPORTED, "xb_create: no kernels for n_base=%d state_len=%d", n_base, state_len);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return xb_fail(nullptr, XB_ERR_CUDA, "xb_create: no CUDA device (%s); this library has no CPU path",
                       cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return xb_fail(nullptr, XB_ERR_ARG, "xb_create: device %d out of range", device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
        return xb_fail(nullptr, XB_ERR_UNSUPPORTED, "xb_create: device %d is not compute capability 10.x (sm_100a only)", device);
    if (cudaSetDevice(device) != cudaSuccess) return xb_fail(nullptr, XB_ERR_CUDA, "cudaSetDevice(%d) failed", device);

    xb_handle *h = new xb_handle();
    h->device = device;
    h->max_N = max_N;
    h->max_T = max_T;
    h->n_base = n_base;
    h->state_len = state_len;
    h->C = ipow(n_base, state_len);
    h->NZ = n_base + 1;
    h->flags = flags;
    h->bf16 = (flags & XB_FLAG_BF16) != 0;
    h->num_sms = prop.multiProcessorCount;
    strncpy(h->alphabet, alphabet, sizeof h->alphabet - 1);

    const size_t TN = (size_t)max_T * max_N, S = (size_t)h->C * h->NZ;
    int rc = XB_OK;
#define TRY(x) if (rc == XB_OK) rc = (x)
    const size_t VP = (size_t)((h->C + 31) / 32) * 32 + 4;
    TRY(dev_alloc(h, &h->alpha, (TN + max_N) * VP));
    TRY(dev_alloc(h, &h->bmax, (TN + max_N) * VP));
    TRY(dev_alloc(h, &h->lp, (TN + max_N) * VP));
    TRY(dev_alloc(h, &h->logz, (size_t)max_N));
    TRY(dev_alloc(h, &h->seq_dev, TN));
    TRY(dev_alloc(h, &h->lens_dev, (size_t)max_N));
    if (!(flags & XB_FLAG_NO_ENCODER)) {
        TRY(dev_alloc_bytes(h, &h->c2, TN * XB_CONV3_K * 2));
        TRY(dev_alloc_bytes(h, &h->act0, TN * XB_FEATURES * 2));
        TRY(dev_alloc_bytes(h, &h->act1, TN * XB_FEATURES * 2));
        TRY(dev_alloc_bytes(h, &h->gates, TN * XB_GATES * 2));
        TRY(dev_alloc(h, &h->cstate, (size_t)max_N * XB_FEATURES));
        TRY(dev_alloc(h, &h->scores, TN * S));
        TRY(dev_alloc_bytes(h, &h->signal_dev, TN * XB_STRIDE * sizeof(float)));
    }
#undef TRY
    if (rc != XB_OK) {
        xb_global_err = h->err;
        xb_destroy(h);
        return rc;
    }
    *out = h;
    return XB_OK;
}

int xb_destroy(xb_handle *h) {
    if (!h) return XB_OK;
    cudaSetDevice(h->device);
    void *ptrs[] = {h->conv1_w, h->conv1_b, h->conv2_w, h->conv2_b, h->conv3_w, h->conv3_b, h->head_w, h->head_b, h->c2,
                    h->act0, h->act1, h->gates, h->cstate, h->hzero, h->scores, h->signal_dev, h->seq_dev, h->lens_dev,
                    h->alpha, h->bmax, h->lp, h->logz, h->ctc_ws, h->lstm_counters};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (void *p : {(void *)h->signal_dev2, (void *)h->seq_dev2, (void *)h->lens_dev2})
        if (p) cudaFree(p);
    if (h->h2d_stream) cudaStreamDestroy(h->h2d_stream);
    if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
    for (int i = 0; i < 2; i++)
        for (cudaEvent_t e : {h->ev_h2d[i], h->ev_enc[i], h->ev_dec[i], h->ev_done[i]})
            if (e) cudaEventDestroy(e);
    for (auto &sp : h->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    for (auto e : h->event_pool) cudaEventDestroy(e);
    for (auto &l : h->lstm) {
        for (void *p : {l.w_ih, l.w_hh, (void *)l.bias, l.w_ihT, l.w_hhT})
            if (p) cudaFree(p);
    }
    if (h->head_wT) cudaFree(h->head_wT);
    if (h->conv3_wT) cudaFree(h->conv3_wT);
    xb_train_free(h);
    delete h;
    return XB_OK;
}

static int alloc_weights(xb_handle *h) {
    if (h->conv1_w) return XB_OK;
    const int F = XB_FEATURES;
    h->head_rows = ipow(h->n_base, h->state_len + 1);
    h->head_rows_padded = ((h->head_rows + 127) / 128) * 128;
    int rc = XB_OK;
#define TRY(x) if (rc == XB_OK) rc = (x)
    TRY(dev_alloc(h, &h->conv1_w, 20));
    TRY(dev_alloc(h, &h->conv1_b, 4));
    TRY(dev_alloc(h, &h->conv2_w, 320));
    TRY(dev_alloc(h, &h->conv2_b, 16));
    TRY(dev_alloc_bytes(h, &h->conv3_w, (size_t)F * XB_CONV3_K * 2));
    TRY(dev_alloc(h, &h->conv3_b, (size_t)F));
    for (auto &l : h->lstm) {
        TRY(dev_alloc_bytes(h, &l.w_ih, (size_t)XB_GATES * F * 2));
        TRY(dev_alloc_bytes(h, &l.w_hh, (size_t)XB_GATES * F * 2));
        TRY(dev_alloc(h, &l.bias, (size_t)XB_GATES));
    }
    TRY(dev_alloc_bytes(h, &h->head_w, (size_t)h->head_rows_padded * F * 2));
    TRY(dev_alloc(h, &h->head_b, (size_t)h->head_rows_padded));
#undef TRY
    return rc;
}

#define XB_WEIGHTS_PROLOGUE()                                                                          \
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");                                        \
    XB_REQUIRE(h, !(h->flags & XB_FLAG_NO_ENCODER), "handle was created with XB_FLAG_NO_ENCODER");     \
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);                                           \
    XB_CUDA(h, cudaSetDevice(h->device));                                                              \
    if (int rc_ = alloc_weights(h)) return rc_

int xb_load_conv_weights(xb_handle *h, const float *w1, const float *b1, const float *w2, const float *b2,
                         const float *w3, const float *b3, void *stream) {
    XB_WEIGHTS_PROLOGUE();
    XB_REQUIRE(h, w1 && b1 && w2 && b2 && w3 && b3, "NULL convolution weight");
    const int F = XB_FEATURES;
    XB_CUDA(h, cudaMemcpyAsync(h->conv1_w, w1, 20 * 4, cudaMemcpyDeviceToDevice, s));
    XB_CUDA(h, cudaMemcpyAsync(h->conv1_b, b1, 4 * 4, cudaMemcpyDeviceToDevice, s));
    XB_CUDA(h, cudaMemcpyAsync(h->conv2_w, w2, 320 * 4, cudaMemcpyDeviceToDevice, s));
    XB_CUDA(h, cudaMemcpyAsync(h->conv2_b, b2, 16 * 4, cudaMemcpyDeviceToDevice, s));
    if (int rc = repack(h, w3, h->conv3_w, F, XB_CONV3_K, F, XB_C2_CH * XB_WINLEN, 2, s)) return rc;
    if (h->flags & XB_FLAG_TRAIN) {
        if (!h->conv3_wT) { if (int rc = dev_alloc_bytes(h, &h->conv3_wT, (size_t)XB_CONV3_K * F * 2)) return rc; }
        if (int rc = repack(h, w3, h->conv3_wT, XB_CONV3_K, F, F, XB_C2_CH * XB_WINLEN, 6, s)) return rc;
    }
    XB_CUDA(h, cudaMemcpyAsync(h->conv3_b, b3, F * 4, cudaMemcpyDeviceToDevice, s));
    h->loaded |= 1;
    return XB_OK;
}

int xb_load_lstm_weights(xb_handle *h, int layer, const float *w_ih, const float *w_hh, const float *b_ih,
                         const float *b_hh, void *stream) {
    XB_WEIGHTS_PROLOGUE();
    XB_REQUIRE(h, layer >= 0 && layer < 5, "LSTM layer %d out of range", layer);
    XB_REQUIRE(h, w_ih && w_hh && b_ih && b_hh, "NULL LSTM weight");
    const int F = XB_FEATURES;
#ifdef XB_EXPERIMENTS
#define XB_FLAG_LSTM_STEPWISE 4
    const int ih_mode = (h->flags & XB_FLAG_LSTM_STEPWISE) ? 1 : 3;
#else
    const int ih_mode = 3;
#endif
    if (int rc = repack(h, w_ih, h->lstm[layer].w_ih, XB_GATES, F, XB_GATES, F, ih_mode, s)) return rc;
    if (int rc = repack(h, w_hh, h->lstm[layer].w_hh, XB_GATES, F, XB_GATES, F, ih_mode == 3 ? 4 : 1, s)) return rc;
    if (h->flags & XB_FLAG_TRAIN) {
        xb_lstm_weights &lw = h->lstm[layer];
        if (!lw.w_ihT) { if (int rc = dev_alloc_bytes(h, &lw.w_ihT, (size_t)XB_GATES * F * 2)) return rc; }
        if (!lw.w_hhT) { if (int rc = dev_alloc_bytes(h, &lw.w_hhT, (size_t)XB_GATES * F * 2)) return rc; }
        if (int rc = repack(h, w_ih, lw.w_ihT, F, XB_GATES, XB_GATES, F, 5, s)) return rc;
        if (int rc = repack(h, w_hh, lw.w_hhT, F, XB_GATES, XB_GATES, F, 5, s)) return rc;
    }
    lstm_bias_kernel<<<(XB_GATES + 255) / 256, 256, 0, s>>>(b_ih, b_hh, h->lstm[layer].bias, ih_mode);
    XB_LAUNCH_CHECK(h);
    h->loaded |= 2 << layer;
    return XB_OK;
}

int xb_load_head_weights(xb_handle *h, const float *w, const float *b, float scale, float blank_score,
                         int expand_blanks, void *stream) {
    XB_WEIGHTS_PROLOGUE();
    XB_REQUIRE(h, w != nullptr, "NULL head weight");
    const int F = XB_FEATURES;
    if (int rc = repack(h, w, h->head_w, h->head_rows_padded, F, h->head_rows, F, 0, s)) return rc;
    if (h->flags & XB_FLAG_TRAIN) {
        if (!h->head_wT) { if (int rc = dev_alloc_bytes(h, &h->head_wT, (size_t)h->head_rows_padded * F * 2)) return rc; }
        if (int rc = repack(h, w, h->head_wT, F, h->head_rows_padded, h->head_rows, F, 5, s)) return rc;
    }
    XB_CUDA(h, cudaMemsetAsync(h->head_b, 0, (size_t)h->head_rows_padded * 4, s));
    if (b) XB_CUDA(h, cudaMemcpyAsync(h->head_b, b, (size_t)h->head_rows * 4, cudaMemcpyDeviceToDevice, s));
    h->scale = scale;
    h->blank_score = blank_score;
    h->expand_blanks = expand_blanks;
    h->loaded |= 64;
    return XB_OK;
}

int xb_load_weights(xb_handle *h, const float *const *w, int n_tensors, float scale, float blank_score, int expand_blanks,
                    void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "xb_load_weights: NULL handle");
    XB_REQUIRE(h, w && n_tensors == XB_NUM_WEIGHTS, "expected %d weight tensors, got %d", XB_NUM_WEIGHTS, n_tensors);
    for (int i = 0; i < n_tensors; i++) XB_REQUIRE(h, w[i] != nullptr, "weight tensor %d is NULL", i);
    if (int rc = xb_load_conv_weights(h, w[0], w[1], w[2], w[3], w[4], w[5], stream)) return rc;
    for (int l = 0; l < 5; l++) {
        const float *const *lw = w + 6 + 4 * l;
        if (int rc = xb_load_lstm_weights(h, l, lw[0], lw[1], lw[2], lw[3], stream)) return rc;
    }
    return xb_load_head_weights(h, w[26], w[27], scale, blank_score, expand_blanks, stream);
}

// ------------------------------------------------------------------------------------------ encoder
}  // extern "C"

// the stem with the masks of dropout sites 0 and 1 (drop may be NULL); the training forward (train_bwd.cu) calls it
int xb_conv_stem_fwd_dropout(xb_handle *h, const void *signal, int sig_dtype, int N, int L, void *out_tnc,
                             const xb_dropout *drop, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    if (!(h->loaded & 1)) return xb_fail(h, XB_ERR_STATE, "convolution weights have not been loaded (xb_load_weights)");
    XB_REQUIRE(h, signal && out_tnc, "NULL buffer");
    XB_REQUIRE(h, L > 0 && L % XB_STRIDE == 0, "chunk length %d must be a positive multiple of the stride %d", L, XB_STRIDE);
    const int T = L / XB_STRIDE;
    if (int rc = check_tn(h, T, N)) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    {
        xb_stage_timer tm(h, XB_ST_CONV12, s);
        if (int rc = xb_conv12_im2col(h, signal, sig_dtype, N, L, s, drop)) return rc;
    }
    xb_stage_timer tm(h, XB_ST_CONV3, s);
    return xb_conv3_launch(h, h->c2, h->conv3_w, h->conv3_b, out_tnc, T, N, s);
}

extern "C" {

int xb_conv_stem_fwd(xb_handle *h, const void *signal, int sig_dtype, int N, int L, void *out_tnc, void *stream) {
    return xb_conv_stem_fwd_dropout(h, signal, sig_dtype, N, L, out_tnc, nullptr, stream);
}

int xb_lstm_fwd(xb_handle *h, int layer, const void *x_tnc, void *y_tnc, int T, int N, int reverse, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, layer >= 0 && layer < 5, "LSTM layer %d out of range", layer);
    if (!(h->loaded & (2 << layer))) return xb_fail(h, XB_ERR_STATE, "weights of LSTM layer %d have not been loaded", layer);
    XB_REQUIRE(h, x_tnc && y_tnc && x_tnc != y_tnc, "x and y must be distinct non-NULL buffers");
    if (int rc = check_tn(h, T, N)) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const xb_lstm_weights &lw = h->lstm[layer];
    // (a) input projection for all time steps: gates (T*N, 3072) = x W_ih^T + (b_ih + b_hh)
    {
        xb_stage_timer tm(h, XB_ST_INPROJ, s);
#ifdef XB_EXPERIMENTS
        static const bool generic = getenv("XB_INPROJ_GENERIC") != nullptr;    // A/B switch: the generic tile kernel
        if (generic) {
            CUtensorMap tmA, tmB;
            if (int rc = xb_make_tmap_2d(h, &tmA, x_tnc, (uint64_t)T * N, XB_FEATURES, XB_FEATURES)) return rc;
            if (int rc = xb_make_tmap_2d(h, &tmB, lw.w_ih, XB_GATES, XB_FEATURES, XB_FEATURES)) return rc;
            GemmParams p;
            p.M = T * N; p.N = XB_GATES; p.K = XB_FEATURES;
            p.bias = lw.bias; p.out = h->gates; p.ldo = XB_GATES;
            if (int rc = xb_gemm_launch(h, EPI_INPROJ, tmA, tmB, p, s)) return rc;
        } else
#endif
        if (int rc = xb_inproj_launch(h, x_tnc, lw.w_ih, lw.bias, h->gates, T * N, s)) return rc;
    }
    // (b) recurrence: one persistent launch per layer; direction by indexing
    xb_stage_timer tm(h, XB_ST_LSTM_REC, s);
#ifdef XB_EXPERIMENTS
    if (h->flags & XB_FLAG_LSTM_STEPWISE) {      // one fused GEMM + cell kernel per time step (independent cross-check)
        CUtensorMap tmH, tmW;
        if (int rc = xb_make_tmap_2d(h, &tmH, y_tnc, (uint64_t)T * N, XB_FEATURES, XB_FEATURES)) return rc;
        if (int rc = xb_make_tmap_2d(h, &tmW, lw.w_hh, XB_GATES, XB_FEATURES, XB_FEATURES)) return rc;
        for (int i = 0; i < T; i++) {
            const int t = reverse ? T - 1 - i : i;
            const int tp = reverse ? t + 1 : t - 1;
            GemmParams p;
            p.M = N; p.N = XB_GATES; p.K = XB_FEATURES;
            p.a_row_offset = (i == 0) ? 0 : tp * N;
            p.out = y_tnc; p.NB = N;
            p.gates = h->gates; p.cstate = h->cstate;
            p.t_cur = t; p.first = (i == 0);
            if (int rc = xb_gemm_launch(h, EPI_LSTM, tmH, tmW, p, s)) return rc;
        }
        return XB_OK;
    }
#endif
    return xb_lstm_recurrence_persistent(h, layer, y_tnc, T, N, reverse, s);
}

int xb_lstm_stack_fwd(xb_handle *h, void *x_tnc, void *y_tnc, int T, int N, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, x_tnc && y_tnc && x_tnc != y_tnc, "x and y must be distinct non-NULL buffers");
    // reverse, forward, reverse, forward, reverse (bonito/crf/model.py:152-154); ping-pong x -> y -> x -> y -> x -> y
    void *a = x_tnc, *b = y_tnc;
    for (int l = 0; l < 5; l++) {
        if (int rc = xb_lstm_fwd(h, l, a, b, T, N, (l % 2) == 0, stream)) return rc;
        void *t = a; a = b; b = t;
    }
    return XB_OK;   // 5 layers: result landed in y_tnc
}

// exp_out: write exp(score) (xb_score_exp) instead of the score -- the hand-over format of the fused host entry points
static int head_fwd(xb_handle *h, const void *x_tnc, float *scores, int T, int N, int exp_out, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    if (!(h->loaded & 64)) return xb_fail(h, XB_ERR_STATE, "CRF head weights have not been loaded (xb_load_weights)");
    XB_REQUIRE(h, x_tnc && scores, "NULL buffer");
    if (int rc = check_tn(h, T, N)) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    xb_stage_timer tm(h, XB_ST_HEAD, s);
#ifdef XB_EXPERIMENTS
    static const bool tile_gemm = getenv("XB_HEAD_GENERIC") != nullptr;      // the 128x128 tile GEMM, kept for cross-checks
    if (tile_gemm) {
        CUtensorMap tmA, tmB;
        if (int rc = xb_make_tmap_2d(h, &tmA, x_tnc, (uint64_t)T * N, XB_FEATURES, XB_FEATURES)) return rc;
        if (int rc = xb_make_tmap_2d(h, &tmB, h->head_w, h->head_rows_padded, XB_FEATURES, XB_FEATURES)) return rc;
        GemmParams p;
        p.M = T * N; p.N = h->head_rows_padded; p.K = XB_FEATURES;
        p.bias = h->head_b; p.out = scores;
        p.ldo = h->expand_blanks ? h->C * h->NZ : h->head_rows;
        p.n_base = h->n_base; p.head_rows = h->head_rows; p.expand = h->expand_blanks;
        p.scale = h->scale; p.blank = h->blank_score;
        return xb_gemm_launch(h, EPI_HEAD, tmA, tmB, p, s);
    }
#endif
    return xb_head_astationary_launch(h, x_tnc, h->head_w, h->head_rows_padded, h->head_b, h->head_rows, scores,
                                      h->expand_blanks ? h->C * h->NZ : h->head_rows, T * N, exp_out, s);
}

int xb_crf_head_fwd(xb_handle *h, const void *x_tnc, float *scores, int T, int N, void *stream) {
    return head_fwd(h, x_tnc, scores, T, N, 0, stream);
}

int xb_crf_head_fwd_exp(xb_handle *h, const void *x_tnc, float *escores, int T, int N, void *stream) {
    if (h && !h->expand_blanks) return xb_fail(h, XB_ERR_STATE, "the exp hand-over format needs expand_blanks");
    return head_fwd(h, x_tnc, escores, T, N, 1, stream);
}

static int encoder_fwd(xb_handle *h, const void *signal, int sig_dtype, int N, int L, float *scores, int exp_out, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, L > 0 && L % XB_STRIDE == 0, "chunk length %d must be a positive multiple of the stride %d", L, XB_STRIDE);
    const int T = L / XB_STRIDE;
    if (int rc = xb_conv_stem_fwd(h, signal, sig_dtype, N, L, h->act0, stream)) return rc;
    if (int rc = xb_lstm_stack_fwd(h, h->act0, h->act1, T, N, stream)) return rc;
    return head_fwd(h, h->act1, scores, T, N, exp_out, stream);
}

int xb_encoder_fwd(xb_handle *h, const void *signal, int sig_dtype, int N, int L, float *scores, void *stream) {
    return encoder_fwd(h, signal, sig_dtype, N, L, scores, 0, stream);
}

// Fused encoder + decode of chunks that are already on the device: the head hands exp(scores) to the decode (h->scores
// never holds log-domain scores on this route), labels / packed rows come back.  The *_host entry points and the read-set
// pipeline run through here.
int xb_basecall_chunks(xb_handle *h, const void *signal, int sig_dtype, int N, int L, int8_t *seq, int8_t *qstring,
                       int32_t *lens, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, signal && seq && lens, "NULL buffer");
    if (!h->scores) return xb_fail(h, XB_ERR_STATE, "handle was created without the encoder");
    XB_REQUIRE(h, h->expand_blanks, "the fused route needs expand_blanks (Viterbi decode over C*NZ scores)");
    if (int rc = encoder_fwd(h, signal, sig_dtype, N, L, h->scores, 1, stream)) return rc;
    return xb_decode_lin(h, h->scores, 1, L / XB_STRIDE, N, nullptr, seq, qstring, lens, nullptr,
                         reinterpret_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------ CRF
#define XB_CRF_PROLOGUE()                                                        \
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");                  \
    XB_REQUIRE(h, scores != nullptr, "scores is NULL");                          \
    if (int rc_ = check_tn(h, T, N)) return rc_;                                 \
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream)

int xb_crf_logz(xb_handle *h, const float *scores, int T, int N, float *logz, void *stream) {
    return xb_crf_logz_s(h, scores, T, N, XB_SEMIRING_LOG, logz, stream);
}

int xb_crf_forward_scores(xb_handle *h, const float *scores, int T, int N, float *alpha, void *stream) {
    return xb_crf_forward_scores_s(h, scores, T, N, XB_SEMIRING_LOG, alpha, stream);
}

int xb_crf_backward_scores(xb_handle *h, const float *scores, int T, int N, float *beta, void *stream) {
    return xb_crf_backward_scores_s(h, scores, T, N, XB_SEMIRING_LOG, beta, stream);
}

#define XB_SEMIRING_CHECK() XB_REQUIRE(h, semiring == XB_SEMIRING_LOG || semiring == XB_SEMIRING_MAX, "unknown semiring %d", semiring)

int xb_crf_logz_s(xb_handle *h, const float *scores, int T, int N, int semiring, float *logz, void *stream) {
    XB_CRF_PROLOGUE();
    XB_SEMIRING_CHECK();
    XB_REQUIRE(h, logz != nullptr, "logz is NULL");
    return xb_decode_alpha(h, scores, T, N, nullptr, logz, semiring == XB_SEMIRING_MAX, s);
}

int xb_crf_forward_scores_s(xb_handle *h, const float *scores, int T, int N, int semiring, float *alpha, void *stream) {
    XB_CRF_PROLOGUE();
    XB_SEMIRING_CHECK();
    XB_REQUIRE(h, alpha != nullptr, "alpha is NULL");
    return xb_decode_alpha(h, scores, T, N, alpha, nullptr, semiring == XB_SEMIRING_MAX, s);
}

int xb_crf_backward_scores_s(xb_handle *h, const float *scores, int T, int N, int semiring, float *beta, void *stream) {
    XB_CRF_PROLOGUE();
    XB_SEMIRING_CHECK();
    XB_REQUIRE(h, beta != nullptr, "beta is NULL");
    return xb_decode_backward(h, scores, T, N, beta, beta, semiring == XB_SEMIRING_MAX ? 1 : 2, s);
}

// posteriors(scores, Max): one-hot at the arg-max edge of the max-marginals of every step (first index on ties).
// edges_nt (N, T) int32 receives the flat edge index c*NZ + k; post (T, N, C*NZ), if given, the one-hot tensor.
int xb_crf_posteriors_max(xb_handle *h, const float *scores, int T, int N, int32_t *edges_nt, float *post, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, edges_nt != nullptr, "edges is NULL");
    if (int rc = xb_decode_backward(h, scores, T, N, h->bmax, nullptr, 1, s)) return rc;
    if (int rc = xb_decode_viterbi_fwd(h, scores, h->bmax, T, N, nullptr, nullptr, nullptr, nullptr, edges_nt, s)) return rc;
    if (post) return xb_onehot_edges(h, edges_nt, T, N, h->C * h->NZ, post, s);
    return XB_OK;
}

int xb_crf_posteriors(xb_handle *h, const float *scores, int T, int N, float *post, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, post != nullptr, "post is NULL");
    return xb_decode_lin(h, scores, 0, T, N, nullptr, nullptr, nullptr, nullptr, post, s);
}

int xb_crf_viterbi(xb_handle *h, const float *scores, int T, int N, int8_t *labels_nt, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, labels_nt != nullptr, "labels is NULL");
    if (int rc = xb_decode_backward(h, scores, T, N, h->bmax, nullptr, 1, s)) return rc;
    return xb_decode_viterbi_fwd(h, scores, h->bmax, T, N, labels_nt, nullptr, nullptr, nullptr, nullptr, s);
}

int xb_crf_decode(xb_handle *h, const float *scores, int T, int N, int8_t *seq, int8_t *qstring, int32_t *lens,
                  int8_t *labels_nt, float *post, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, seq != nullptr && lens != nullptr, "seq / lens is NULL");
    return xb_decode_lin(h, scores, 0, T, N, labels_nt, seq, qstring, lens, post, s);
}

// Beam-search decode (csrc/beam_search.cu): Log-semiring backward scores into handle workspace, then the beam
int xb_crf_beam_search(xb_handle *h, const float *scores, int T, int N, int beam_width, float beam_cut, int8_t *seq,
                       int8_t *qstring, int8_t *moves, int32_t *lens, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, seq != nullptr && lens != nullptr, "seq / lens is NULL");
    if (int rc = xb_decode_backward(h, scores, T, N, nullptr, h->lp, 2, s)) return rc;
    return xb_beam_search_impl(h, scores, h->lp, T, N, beam_width, beam_cut, seq, qstring, moves, lens, s);
}

int xb_crf_decode_exp(xb_handle *h, const float *scores, int T, int N, int8_t *seq, int8_t *qstring, int32_t *lens,
                      int8_t *labels_nt, float *post, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, seq != nullptr && lens != nullptr, "seq / lens is NULL");
    return xb_decode_lin(h, scores, 1, T, N, labels_nt, seq, qstring, lens, post, s);
}

int xb_ctc_crf_loss_fwd(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                        const int32_t *lengths, int normalise, float *loss, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, targets && lengths && loss, "NULL buffer");
    return xb_ctc_loss_impl(h, scores, T, N, targets, Lmax, lengths, normalise, loss, s);
}

int xb_ctc_crf_loss_bwd(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                        const int32_t *lengths, int normalise, const float *grad_loss, float *alpha_ws,
                        float *grad_scores, void *stream) {
    XB_CRF_PROLOGUE();
    XB_REQUIRE(h, targets && lengths && grad_loss && alpha_ws && grad_scores, "NULL buffer");
    if (normalise) {       // logZ (for the shift) and the posteriors of the full lattice, straight into grad_scores
        if (int rc = xb_decode_lin(h, scores, 0, T, N, nullptr, nullptr, nullptr, nullptr, grad_scores, s)) return rc;
        if (int rc = xb_decode_alpha(h, scores, T, N, nullptr, h->logz, 0, s)) return rc;
    }
    return xb_ctc_loss_bwd_impl(h, scores, T, N, targets, Lmax, lengths, normalise, grad_loss, alpha_ws, grad_scores, s);
}

int xb_stitch(xb_handle *h, const int8_t *rows, int T, const int32_t *chunk_first, const int32_t *chunk_count,
              const int32_t *read_len, int n_reads, int chunksize, int overlap, int stride, int reverse, int8_t *out,
              int out_stride, int32_t *out_len, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, rows && chunk_first && chunk_count && read_len && out && out_len, "NULL buffer");
    XB_CUDA(h, cudaSetDevice(h->device));
    return xb_stitch_impl(h, rows, T, chunk_first, chunk_count, read_len, n_reads, chunksize, overlap, stride, reverse, out,
                          out_stride, out_len, reinterpret_cast<cudaStream_t>(stream));
}

int xb_gather_chunks(xb_handle *h, const void *signal, int sig_dtype, const int64_t *read_offset, const int32_t *read_len,
                     const int32_t *chunk_read, const int32_t *chunk_start, int n_chunks, int L, float *out, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, signal && read_offset && read_len && chunk_read && chunk_start && out, "NULL buffer");
    XB_CUDA(h, cudaSetDevice(h->device));
    return xb_gather_chunks_impl(h, signal, sig_dtype, read_offset, read_len, chunk_read, chunk_start, n_chunks, L, out,
                                 reinterpret_cast<cudaStream_t>(stream));
}

int xb_preprocess_reads(xb_handle *h, const int16_t *raw, const int64_t *read_offset, const int32_t *read_len,
                        const double *scaling, const int32_t *offset, int n_reads, float *out, int32_t *out_len,
                        float *stats, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, raw && read_offset && read_len && scaling && offset && out && out_len && stats, "NULL buffer");
    XB_CUDA(h, cudaSetDevice(h->device));
    return xb_preprocess_impl(h, raw, read_offset, read_len, scaling, offset, n_reads, out, out_len, stats,
                              reinterpret_cast<cudaStream_t>(stream));
}

int xb_compute_scores_host(xb_handle *h, const float *signal_host, int N, int L, int8_t *seq_host, int32_t *lens_host,
                           void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, signal_host && seq_host && lens_host, "NULL buffer");
    XB_REQUIRE(h, L > 0 && L % XB_STRIDE == 0, "chunk length %d must be a positive multiple of the stride %d", L, XB_STRIDE);
    const int T = L / XB_STRIDE;
    if (int rc = check_tn(h, T, N)) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    XB_CUDA(h, cudaMemcpyAsync(h->signal_dev, signal_host, (size_t)N * L * sizeof(float), cudaMemcpyHostToDevice, s));
    if (int rc = xb_basecall_chunks(h, h->signal_dev, XB_SIG_F32, N, L, h->seq_dev, nullptr, h->lens_dev, stream)) return rc;
    XB_CUDA(h, cudaMemcpyAsync(seq_host, h->seq_dev, (size_t)N * T, cudaMemcpyDeviceToHost, s));
    XB_CUDA(h, cudaMemcpyAsync(lens_host, h->lens_dev, (size_t)N * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    XB_CUDA(h, cudaStreamSynchronize(s));
    return XB_OK;
}

// Pipelined form of xb_compute_scores_host: two slots; submit() enqueues H2D (own copy stream), encoder + decode (the
// caller's stream) and D2H (second copy stream) of one batch and returns, wait() blocks until the slot's results are in
// the host buffers.  With batch i+1 submitted before batch i is awaited, the copies of one batch hide under the kernels
// of the other.  A slot must be awaited before it is submitted again; host buffers must stay valid until then.
static int pipeline_init(xb_handle *h) {
    if (h->h2d_stream) return XB_OK;
    const size_t TN = (size_t)h->max_T * h->max_N;
    XB_CUDA(h, cudaMalloc(&h->signal_dev2, TN * XB_STRIDE * sizeof(float)));
    XB_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&h->seq_dev2), TN));
    XB_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&h->lens_dev2), (size_t)h->max_N * sizeof(int32_t)));
    XB_CUDA(h, cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking));
    XB_CUDA(h, cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        XB_CUDA(h, cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
        XB_CUDA(h, cudaEventCreateWithFlags(&h->ev_enc[i], cudaEventDisableTiming));
        XB_CUDA(h, cudaEventCreateWithFlags(&h->ev_dec[i], cudaEventDisableTiming));
        XB_CUDA(h, cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
    }
    return XB_OK;
}

int xb_compute_scores_submit(xb_handle *h, int slot, const float *signal_host, int N, int L, int8_t *seq_host,
                             int32_t *lens_host, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, slot == 0 || slot == 1, "slot must be 0 or 1");
    XB_REQUIRE(h, signal_host && seq_host && lens_host, "NULL buffer");
    XB_REQUIRE(h, L > 0 && L % XB_STRIDE == 0, "chunk length %d must be a positive multiple of the stride %d", L, XB_STRIDE);
    const int T = L / XB_STRIDE;
    if (int rc = check_tn(h, T, N)) return rc;
    if (!h->signal_dev) return xb_fail(h, XB_ERR_STATE, "handle was created without the encoder");
    if (int rc = pipeline_init(h)) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    void *sig = slot ? h->signal_dev2 : h->signal_dev;
    int8_t *seq = slot ? h->seq_dev2 : h->seq_dev;
    int32_t *lens = slot ? h->lens_dev2 : h->lens_dev;
    if (h->slot_used[slot]) {       // the slot's previous batch: its signal has been consumed, its results have left
        XB_CUDA(h, cudaStreamWaitEvent(h->h2d_stream, h->ev_enc[slot], 0));
        XB_CUDA(h, cudaStreamWaitEvent(s, h->ev_done[slot], 0));
    }
    XB_CUDA(h, cudaMemcpyAsync(sig, signal_host, (size_t)N * L * sizeof(float), cudaMemcpyHostToDevice, h->h2d_stream));
    XB_CUDA(h, cudaEventRecord(h->ev_h2d[slot], h->h2d_stream));
    XB_CUDA(h, cudaStreamWaitEvent(s, h->ev_h2d[slot], 0));
    if (int rc = encoder_fwd(h, sig, XB_SIG_F32, N, L, h->scores, 1, stream)) return rc;
    XB_CUDA(h, cudaEventRecord(h->ev_enc[slot], s));
    if (int rc = xb_decode_lin(h, h->scores, 1, T, N, nullptr, seq, nullptr, lens, nullptr, s)) return rc;
    XB_CUDA(h, cudaEventRecord(h->ev_dec[slot], s));
    XB_CUDA(h, cudaStreamWaitEvent(h->d2h_stream, h->ev_dec[slot], 0));
    XB_CUDA(h, cudaMemcpyAsync(seq_host, seq, (size_t)N * T, cudaMemcpyDeviceToHost, h->d2h_stream));
    XB_CUDA(h, cudaMemcpyAsync(lens_host, lens, (size_t)N * sizeof(int32_t), cudaMemcpyDeviceToHost, h->d2h_stream));
    XB_CUDA(h, cudaEventRecord(h->ev_done[slot], h->d2h_stream));
    h->slot_used[slot] = true;
    return XB_OK;
}

int xb_compute_scores_wait(xb_handle *h, int slot) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, (slot == 0 || slot == 1) && h->slot_used[slot], "slot %d has nothing in flight", slot);
    XB_CUDA(h, cudaSetDevice(h->device));
    XB_CUDA(h, cudaEventSynchronize(h->ev_done[slot]));
    return XB_OK;
}

int xb_gemm_selftest(xb_handle *h, const void *A, const void *B, float *D, int M, int N, int K, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, A && B && D && M > 0 && N > 0 && K > 0, "bad GEMM arguments");
    CUtensorMap tmA, tmB;
    if (int rc = xb_make_tmap_2d(h, &tmA, A, M, K, K)) return rc;
    if (int rc = xb_make_tmap_2d(h, &tmB, B, N, K, K)) return rc;
    GemmParams p;
    p.M = M; p.N = N; p.K = K; p.out = D; p.ldo = N;
    return xb_gemm_launch(h, EPI_F32, tmA, tmB, p, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
