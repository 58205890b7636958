// Per-read signal pre-processing on the GPU (SURVEY section 8f, N2): int16 DAC values -> pA scaling -> trim of the
// leading stall -> med/MAD normalisation, i.e. what the reference does per read on the CPU inside an 8-process pool
// (ub-bonito/bonito/fast5.py: Read.__init__ :88-100, trim :149-172; bonito/util.py med_mad, norm_by_noisiest_section).
//
// One CTA per read.  Every quantity the reference derives from order statistics (medians) is computed exactly with an
// 8-bit radix select over order-preserving keys, every float32 operation is spelled with round-to-nearest intrinsics in
// the order numpy evaluates it, and the two float32 reductions of the short-read branch (np.std) replay numpy's pairwise
// summation tree -- so the normalised signal has the same bits as the reference's (checked against oracle/preprocess.py,
// which is pinned against the reference's own functions).  The scaled signal is never stored: it is recomputed from the
// int16 samples (2 bytes each, L1/L2-resident for the ~10 passes of a read) wherever it is needed.
#include <float.h>

#include "xb_common.cuh"

namespace {

constexpr int PP_THREADS = 256;
constexpr int PP_HEAD = 8000;        // samples trim() looks at; reads no longer than this use the noisiest section
constexpr int PP_MIN_TRIM = 10, PP_TRIM_WINDOW = 40, PP_TRIM_TAIL = 4000, PP_NOISE_WINDOW = 100;

__device__ __forceinline__ uint32_t fkey(float x) {
    const uint32_t b = __float_as_uint(x);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float keyf(uint32_t k) {
    return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu));
}

struct ScaledRead {                  // fast5.py:88-89: float32(scaling * (raw + offset)), product in float64
    const int16_t *raw;
    double scaling;
    int offset;
    __device__ __forceinline__ float operator()(int i) const {
        return (float)(scaling * (double)((int)raw[i] + offset));
    }
};

struct Scratch {
    uint32_t hist[256];
    uint32_t bc[4];
};

// k-th smallest (0-based) key among key(0..n-1); called by the whole CTA, result returned to every thread.
template <class KeyFn> __device__ uint32_t block_select(KeyFn key, int n, int k, Scratch &sc) {
    uint32_t prefix = 0, mask = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int b = threadIdx.x; b < 256; b += blockDim.x) sc.hist[b] = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const uint32_t kk = key(i);
            if ((kk & mask) == prefix) atomicAdd(&sc.hist[(kk >> shift) & 255], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t cum = 0;
            int b = 0;
            for (; b < 255; b++) {
                if (cum + sc.hist[b] > (uint32_t)k) break;
                cum += sc.hist[b];
            }
            sc.bc[0] = (uint32_t)b;
            sc.bc[1] = cum;
        }
        __syncthreads();
        prefix |= sc.bc[0] << shift;
        mask |= 255u << shift;
        k -= (int)sc.bc[1];
        __syncthreads();
    }
    return prefix;
}

// np.median of float32 values: the middle element, or the float32 mean of the two middle elements.
template <class KeyFn> __device__ float block_median(KeyFn key, int n, Scratch &sc) {
    if (n & 1) return keyf(block_select(key, n, n / 2, sc));
    const uint32_t v0 = block_select(key, n, n / 2 - 1, sc);
    if (threadIdx.x == 0) { sc.bc[2] = 0u; sc.bc[3] = 0xffffffffu; }
    __syncthreads();
    uint32_t le = 0, mn = 0xffffffffu;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const uint32_t kk = key(i);
        if (kk <= v0) le++;
        else mn = min(mn, kk);
    }
    atomicAdd(&sc.bc[2], le);
    atomicMin(&sc.bc[3], mn);
    __syncthreads();
    const uint32_t v1 = (sc.bc[2] > (uint32_t)(n / 2)) ? v0 : sc.bc[3];
    __syncthreads();
    return __fmul_rn(__fadd_rn(keyf(v0), keyf(v1)), 0.5f);
}

// numpy's pairwise float32 summation (umath loops_utils: 8 accumulators on blocks of <= 128, halves rounded down to a
// multiple of 8 above that), over f(lo .. lo+n-1); one thread.
template <class F> __device__ float np_pairwise_sum(F f, int lo, int n) {
    if (n < 8) {
        float res = 0.0f;
        for (int i = 0; i < n; i++) res = __fadd_rn(res, f(lo + i));
        return res;
    }
    if (n <= 128) {
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = f(lo + j);
        int i = 8;
        for (; i < n - (n % 8); i += 8)
#pragma unroll
            for (int j = 0; j < 8; j++) r[j] = __fadd_rn(r[j], f(lo + i + j));
        float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                              __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
        for (; i < n; i++) res = __fadd_rn(res, f(lo + i));
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    const float a = np_pairwise_sum(f, lo, n2);
    const float b = np_pairwise_sum(f, lo + n2, n - n2);
    return __fadd_rn(a, b);
}

// np.std of a float32 array (ddof 0): mean, squared deviations and their mean in float32, pairwise sums; one thread.
__device__ float np_std(const float *a, int n) {
    const float fn = (float)n;
    const float mean = __fdiv_rn(__fadd_rn(0.0f, np_pairwise_sum([&](int i) { return a[i]; }, 0, n)), fn);
    const float ss = np_pairwise_sum([&](int i) { const float d = __fsub_rn(a[i], mean); return __fmul_rn(d, d); }, 0, n);
    return __fsqrt_rn(__fdiv_rn(__fadd_rn(0.0f, ss), fn));
}

__device__ __forceinline__ float mad_from_median(float mm) {      // util.med_mad: median(|x - med|) * 1.4826 + eps
    return __fadd_rn(__fmul_rn(mm, 1.4826f), FLT_EPSILON);
}

__global__ void __launch_bounds__(PP_THREADS)
preprocess_kernel(const int16_t *__restrict__ raw_all, const int64_t *__restrict__ read_offset,
                  const int32_t *__restrict__ read_len, const double *__restrict__ scaling,
                  const int32_t *__restrict__ offset, float *__restrict__ out_all, int32_t *__restrict__ out_len,
                  float *__restrict__ stats) {
    __shared__ Scratch sc;
    __shared__ float sbuf[PP_HEAD];
    __shared__ unsigned char wflag[PP_HEAD / PP_TRIM_WINDOW];
    __shared__ float wstd[PP_HEAD / PP_NOISE_WINDOW];
    __shared__ float thr_s;
    __shared__ int res_s[2];
    const int r = blockIdx.x, tid = threadIdx.x;
    const ScaledRead src{raw_all + read_offset[r], scaling[r], offset[r]};
    const int len = read_len[r];
    float *out = out_all + read_offset[r];

    // ---- trim (fast5.py:149-172) on scaled[:8000]
    const int head = min(len, PP_HEAD), L = max(head - PP_MIN_TRIM, 0);
    int start = PP_MIN_TRIM;
    if (L > 0) {
        const int wn = min(L, PP_TRIM_TAIL), w0 = PP_MIN_TRIM + (L - wn);
        const float med = block_median([&](int i) { return fkey(src(w0 + i)); }, wn, sc);
        const float mm = block_median([&](int i) { return fkey(fabsf(__fsub_rn(src(w0 + i), med))); }, wn, sc);
        const float thr = __fadd_rn(med, __fmul_rn(mad_from_median(mm), 2.4f));
        const int nw = L / PP_TRIM_WINDOW;
        for (int p = tid; p < nw; p += PP_THREADS) {
            int cnt = 0;
            bool last = false;
            for (int q = 0; q < PP_TRIM_WINDOW; q++) {
                last = src(PP_MIN_TRIM + p * PP_TRIM_WINDOW + q) > thr;
                cnt += last;
            }
            wflag[p] = (unsigned char)((cnt > 3 ? 1 : 0) | (last ? 2 : 0));
        }
        __syncthreads();
        if (tid == 0) {
            bool seen = false;
            int res = PP_MIN_TRIM;
            for (int pos = 0; pos < nw; pos++) {
                if ((wflag[pos] & 1) || seen) {
                    seen = true;
                    if (wflag[pos] & 2) continue;
                    res = min((pos + 1) * PP_TRIM_WINDOW + PP_MIN_TRIM, L);
                    break;
                }
            }
            res_s[0] = res;
        }
        __syncthreads();
        start = res_s[0];
    }
    const int n2 = len - start;
    if (n2 <= 0) {
        if (tid == 0) {
            out_len[r] = 0;
            stats[r * 4 + 0] = (float)start; stats[r * 4 + 1] = 0.0f; stats[r * 4 + 2] = 0.0f; stats[r * 4 + 3] = 2.0f;
        }
        return;
    }

    float med, mad;
    const bool is_short = n2 <= PP_HEAD;
    if (!is_short) {
        med = block_median([&](int i) { return fkey(src(start + i)); }, n2, sc);
        mad = mad_from_median(block_median([&](int i) { return fkey(fabsf(__fsub_rn(src(start + i), med))); }, n2, sc));
    } else {
        // ---- norm_by_noisiest_section: windows of 100 samples whose std exceeds std(signal) / 6 are "noisy"; the med/MAD
        // come from the longest run of noisy samples (plus the sample before it), the whole signal if there is none
        for (int i = tid; i < n2; i += PP_THREADS) sbuf[i] = src(start + i);
        __syncthreads();
        const int nwin = n2 / PP_NOISE_WINDOW;
        if (tid == 0) thr_s = __fdiv_rn(np_std(sbuf, n2), 6.0f);
        if (tid >= 32 && tid - 32 < nwin) wstd[tid - 32] = np_std(sbuf + (tid - 32) * PP_NOISE_WINDOW, PP_NOISE_WINDOW);
        __syncthreads();
        if (tid == 0) {
            int best_a = 0, best_b = n2, best_len = 0, run0 = -1;
            for (int i = 0; i <= n2; i++) {
                bool one = false;
                if (i > 0 && i < n2 - 1) one = (i < nwin * PP_NOISE_WINDOW) ? (wstd[i / PP_NOISE_WINDOW] > thr_s) : true;
                if (one) {
                    if (run0 < 0) run0 = i;
                } else if (run0 >= 0) {
                    if (i - run0 > best_len) { best_len = i - run0; best_a = run0 - 1; best_b = i; }
                    run0 = -1;
                }
            }
            res_s[0] = best_a;
            res_s[1] = best_b;
        }
        __syncthreads();
        const int a = res_s[0], cnt = res_s[1] - res_s[0];
        med = block_median([&](int i) { return fkey(sbuf[a + i]); }, cnt, sc);
        mad = mad_from_median(block_median([&](int i) { return fkey(fabsf(__fsub_rn(sbuf[a + i], med))); }, cnt, sc));
    }
    for (int i = tid; i < n2; i += PP_THREADS)
        out[i] = __fdiv_rn(__fsub_rn(is_short ? sbuf[i] : src(start + i), med), mad);
    if (tid == 0) {
        out_len[r] = n2;
        stats[r * 4 + 0] = (float)start; stats[r * 4 + 1] = med; stats[r * 4 + 2] = mad; stats[r * 4 + 3] = is_short ? 1.0f : 0.0f;
    }
}

}  // namespace

extern "C" int xb_preprocess_reads(xb_handle *h, const int16_t *raw, const int64_t *read_offset, const int32_t *read_len,
                                   const double *scaling, const int32_t *offset, int n_reads, float *out, int32_t *out_len,
                                   float *stats, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, raw && read_offset && read_len && scaling && offset && out && out_len && stats, "NULL buffer");
    XB_CUDA(h, cudaSetDevice(h->device));
    XB_REQUIRE(h, n_reads > 0, "bad pre-processing arguments");
    preprocess_kernel<<<n_reads, PP_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(raw, read_offset, read_len, scaling,
                                                                                         offset, out, out_len, stats);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
