// Shared internals of libxna_b200.so: handle, error plumbing, small device helpers.
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/xna_basecaller.h"

#define XB_FEATURES 768          // encoder width of the sup@v3.3 architecture (config.toml [encoder] features)
#define XB_GATES (4 * XB_FEATURES)
#define XB_STRIDE 5
#define XB_WINLEN 19
#define XB_C2_CH 16              // channels after the second convolution
#define XB_C2_HALO 9             // winlen // 2
#define XB_CONV3_K 320           // 19*16 = 304 padded to a multiple of 64 (zero weights)
#define XB_LSTM_COUNTERS 2048    // ints of the persistent LSTM kernel's step counters (lstm_persistent.cu MAX_CTRS x CTR_STRIDE)

struct xb_lstm_weights {
    void *w_ih = nullptr;        // (3072, 768) 16-bit, rows gate-interleaved (see xb_api.cu)
    void *w_hh = nullptr;        // (3072, 768) 16-bit, same row order
    float *bias = nullptr;       // (3072) fp32 = b_ih + b_hh, same row order
    void *w_ihT = nullptr;       // XB_FLAG_TRAIN: (768, 3072) bf16 = W_ih^T, reference gate-row order (backward GEMM operand)
    void *w_hhT = nullptr;       // XB_FLAG_TRAIN: (768, 3072) bf16 = W_hh^T
};

enum { XB_ST_CONV12 = 0, XB_ST_CONV3, XB_ST_INPROJ, XB_ST_LSTM_REC, XB_ST_HEAD, XB_ST_CRF_ALPHA, XB_ST_CRF_BACKWARD,
       XB_ST_CRF_VITERBI, XB_ST_TRAIN_BPTT, XB_ST_TRAIN_TRANSPOSE, XB_ST_TRAIN_WGRAD, XB_ST_TRAIN_XGRAD, XB_ST_TRAIN_HEAD_CONV,
       XB_ST_COUNT };

struct xb_prof_span { int stage; cudaEvent_t a, b; };

struct xb_handle {
    int device = 0;
    bool profiling = false;
    std::vector<xb_prof_span> spans;
    std::vector<cudaEvent_t> event_pool;
    int max_N = 0, max_T = 0;
    int n_base = 0, state_len = 0, C = 0, NZ = 0;
    int flags = 0;
    bool bf16 = false;
    int loaded = 0;              // bit 0 conv stem, bits 1..5 LSTM layers, bit 6 CRF head
    char alphabet[16] = {0};
    int num_sms = 0;
    int64_t launches = 0;
    std::string err;

    // weights (device)
    float *conv1_w = nullptr, *conv1_b = nullptr, *conv2_w = nullptr, *conv2_b = nullptr;
    void *conv3_w = nullptr;     // (768, 320) 16-bit: k = tap*16 + channel, zero padded
    float *conv3_b = nullptr;
    xb_lstm_weights lstm[5];
    void *head_w = nullptr;      // (head_rows_padded, 768) 16-bit
    float *head_b = nullptr;
    int head_rows = 0, head_rows_padded = 0;
    float scale = 5.0f, blank_score = 2.0f;
    int expand_blanks = 1;

    // encoder workspace
    void *c2 = nullptr;          // (max_N, L + 2*halo (+pad), 16) 16-bit channel-last conv2 output
    void *act0 = nullptr, *act1 = nullptr;   // (max_T, max_N, 768) 16-bit ping-pong
    void *gates = nullptr;       // (max_T, max_N, 3072) 16-bit hoisted input projection
    float *scores = nullptr;     // (max_T, max_N, C*NZ) fp32 (used by the host entry points)
    int *lstm_counters = nullptr; // XB_LSTM_COUNTERS per-group step counters of the persistent LSTM kernel
    // the two slots of the host entry points (xb_compute_scores_submit / _wait): slot 0 is allocated with the encoder
    // workspace, slot 1, the copy streams and the events on first use
    void *signal_dev[2] = {};    // (max_N, max_T*5) fp32 staging
    int8_t *seq_dev[2] = {};     // (max_N, max_T)
    int32_t *lens_dev[2] = {};   // (max_N)
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_enc[2] = {nullptr, nullptr}, ev_dec[2] = {nullptr, nullptr},
                ev_done[2] = {nullptr, nullptr};
    bool slot_used[2] = {false, false};

    // decode workspace
    // three (max_T+1, max_N, VP) state-vector buffers, VP = round_up(C, 32) + 4 floats (16-byte aligned rows for the
    // bulk-copy ring of crf_decode_lin.cu); the log-domain scans use them with pitch C
    float *alpha = nullptr;      // linear decode: a_hat;  log-domain scans: alpha
    float *bmax = nullptr;       // linear decode: bm_hat; log-domain scans: Max-semiring beta
    float *beta = nullptr;       // linear decode: b_hat;  beam search: Log-semiring beta
    float *logz = nullptr;       // (max_N)

    // training (XB_FLAG_TRAIN; workspace allocated by the first xb_encoder_fwd_train, see train_bwd.cu)
    void *head_wT = nullptr;     // (768, head_rows_padded) bf16 = W_head^T
    void *conv3_wT = nullptr;    // (320, 768) bf16 = W_3^T in im2col column order
    struct xb_train_ws *train = nullptr;

    // driver entry point for TMA descriptors (resolved at run time: no link-time libcuda dependency)
    void *encode_tiled = nullptr;
    // largest dynamic shared-memory size set per kernel on this handle (xb_smem_attr)
    std::unordered_map<const void *, size_t> smem_attr;
};

extern thread_local std::string xb_global_err;

// CUDA-event span around a stage on the launching stream (only when xb_set_profiling(h, 1))
struct xb_stage_timer {
    xb_handle *h; cudaStream_t s; int idx = -1;
    xb_stage_timer(xb_handle *h_, int stage, cudaStream_t s_) : h(h_), s(s_) {
        if (!h->profiling) return;
        auto get = [&]() { cudaEvent_t e; if (!h->event_pool.empty()) { e = h->event_pool.back(); h->event_pool.pop_back(); }
                           else cudaEventCreate(&e); return e; };
        xb_prof_span sp{stage, get(), get()};
        cudaEventRecord(sp.a, s);
        h->spans.push_back(sp);
        idx = (int)h->spans.size() - 1;
    }
    ~xb_stage_timer() { if (idx >= 0) cudaEventRecord(h->spans[idx].b, s); }
};

int xb_fail(xb_handle *h, int code, const char *fmt, ...);

#define XB_CUDA(h, call)                                                                         \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return xb_fail((h), XB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                           __FILE__, __LINE__);                                                  \
    } while (0)

#define XB_LAUNCH_CHECK(h)                                                                       \
    do {                                                                                         \
        (h)->launches++;                                                                         \
        cudaError_t e_ = cudaGetLastError();                                                     \
        if (e_ != cudaSuccess)                                                                   \
            return xb_fail((h), XB_ERR_CUDA, "kernel launch failed: %s (%s:%d)",                 \
                           cudaGetErrorString(e_), __FILE__, __LINE__);                          \
    } while (0)

#define XB_REQUIRE(h, cond, ...)                                                                 \
    do {                                                                                         \
        if (!(cond)) return xb_fail((h), XB_ERR_ARG, __VA_ARGS__);                               \
    } while (0)

// *p = cudaMalloc(bytes) unless *p is already set: allocating a set of buffers through this again after a failure
// completes the set
inline int xb_alloc(xb_handle *h, void **p, size_t bytes) {
    if (*p) return XB_OK;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) return xb_fail(h, XB_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    return XB_OK;
}

// Allows `kernel` `bytes` of dynamic shared memory.  Above the default 48 KB the limit is a function attribute of the
// device's context; the handle records the largest size it has set per kernel, so the attribute is set once per size
// step instead of per launch, and never lowered below what another handle on the same device has set.
template <typename K> int xb_smem_attr(xb_handle *h, K kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return XB_OK;
    size_t &set = h->smem_attr[reinterpret_cast<const void *>(kernel)];
    if (bytes <= set) return XB_OK;
    cudaFuncAttributes fa;
    XB_CUDA(h, cudaFuncGetAttributes(&fa, kernel));
    if ((size_t)fa.maxDynamicSharedSizeBytes > bytes) bytes = fa.maxDynamicSharedSizeBytes;
    XB_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    set = bytes;
    return XB_OK;
}

// ---- 16-bit type helpers (fp16 default, bf16 with XB_FLAG_BF16) ---------------------------------
template <bool BF16> struct xb16;
template <> struct xb16<false> {
    using T = __half;
    using T2 = __half2;
    static __device__ __forceinline__ T from(float x) { return __float2half_rn(x); }
    static __device__ __forceinline__ float to(T x) { return __half2float(x); }
    static __device__ __forceinline__ uint32_t pack(float lo, float hi) {
        __half2 v = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&v);
    }
    static __device__ __forceinline__ float2 unpack(uint32_t u) {
        return __half22float2(*reinterpret_cast<__half2 *>(&u));
    }
};
template <> struct xb16<true> {
    using T = __nv_bfloat16;
    using T2 = __nv_bfloat162;
    static __device__ __forceinline__ T from(float x) { return __float2bfloat16_rn(x); }
    static __device__ __forceinline__ float to(T x) { return __bfloat162float(x); }
    static __device__ __forceinline__ uint32_t pack(float lo, float hi) {
        __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&v);
    }
    static __device__ __forceinline__ float2 unpack(uint32_t u) {
        return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162 *>(&u));
    }
};

// ---- functions one translation unit defines and others call ------------------------------------------
struct xb_dropout;
// xb_api.cu
int xb_conv_stem_fwd_dropout(xb_handle *h, const void *signal, int sig_dtype, int N, int L, void *out_tnc,
                             const xb_dropout *drop, void *stream);
// conv_stem.cu
int xb_conv12_im2col(xb_handle *h, const void *signal, int sig_dtype, int N, int L, cudaStream_t s,
                     const xb_dropout *drop = nullptr);
// lstm_persistent.cu
int xb_lstm_recurrence_persistent(xb_handle *h, int layer, void *y_tnc, int T, int N, int reverse, cudaStream_t s,
                                  void *save = nullptr);
// inproj_gemm.cu
int xb_inproj_launch(xb_handle *h, const void *x, const void *w_ih, const float *bias, void *gates, int M, cudaStream_t s);
int xb_head_astationary_launch(xb_handle *h, const void *x, const void *w, int w_rows, const float *bias, int head_rows,
                               float *scores, int ldo, int M, int exp_out, cudaStream_t s);
// wgrad_gemm.cu
int xb_lstm_wgrad_launch(xb_handle *h, const void *dzT, const void *xT, const void *yT, int T, int N, bool reverse, float *g_wih,
                         float *g_whh, cudaStream_t s);
// train_bwd.cu
void xb_train_free(xb_handle *h);
// misc_kernels.cu
int xb_onehot_edges(xb_handle *h, const int32_t *edges_nt, int T, int N, int S, float *post, cudaStream_t s);
int xb_ctc_loss_impl(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                     const int32_t *lengths, int normalise, float *loss, cudaStream_t s);
int xb_ctc_loss_bwd_impl(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                         const int32_t *lengths, int normalise, const float *grad_loss, float *alpha_ws, float *grad,
                         cudaStream_t s);
// beam_search.cu
int xb_beam_search_impl(xb_handle *h, const float *scores, const float *beta, int T, int N, int beam_width, float beam_cut,
                        int8_t *seq, int8_t *qstring, int8_t *moves, int32_t *lens, cudaStream_t s);
// crf_decode.cu, crf_decode_lin.cu
int xb_decode_alpha(xb_handle *h, const float *scores, int T, int N, float *alpha, float *logz, int use_max, cudaStream_t s);
int xb_decode_backward(xb_handle *h, const float *scores, int T, int N, float *bmax, float *beta, int mode, cudaStream_t s);
int xb_decode_lin(xb_handle *h, const float *scores, int lin_input, int T, int N, int8_t *labels, int8_t *seq, int8_t *qs,
                  int32_t *lens, float *post, cudaStream_t s);
int xb_decode_viterbi_fwd(xb_handle *h, const float *scores, const float *bmax, int T, int N, int8_t *labels, int32_t *edges,
                          cudaStream_t s);
