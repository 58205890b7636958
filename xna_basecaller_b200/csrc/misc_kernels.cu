// Overlap stitching of left-packed chunk rows and the CTC-CRF training loss forward.
//
//   stitch:   bonito/util.py:169-188 (stitch) applied by bonito/crf/basecall.py:15-24 (stitch_results) to the
//             left-packed (n_chunks, T) int8 rows of compute_scores, followed by koi.decode.to_str
//             (crf/basecall.py:85-93): zeros dropped.  Slices act on ROW POSITIONS of the packed rows -- the
//             reference's behaviour, kept on purpose (SURVEY.md 8a-11).
//   ctc loss: CTC_CRF.ctc_loss / normalise / prepare_ctc_scores (bonito/crf/model.py:48-49,102-131) with
//             seqdist.ctc_simple.logZ_cupy restated as a stay/move lattice scan.
#include "xb_common.cuh"
#include "xb_exact_math.h"

namespace {

// one warp per read
__global__ void stitch_kernel(const int8_t *__restrict__ rows, int T, const int32_t *__restrict__ chunk_first,
                              const int32_t *__restrict__ chunk_count, const int32_t *__restrict__ read_len, int n_reads,
                              int chunksize, int overlap, int stride, int reverse, int8_t *__restrict__ out, int out_stride,
                              int32_t *__restrict__ out_len) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= n_reads) return;
    const int nch = chunk_count[r], first = chunk_first[r], length = read_len[r];
    const int semi = overlap / 2;
    const int start = semi / stride, end = (chunksize - semi) / stride;
    const int stub = (length - overlap) % (chunksize - overlap);
    const int first_end = stub > 0 ? (stub + semi) / stride : end;
    int8_t *o = out + (size_t)r * out_stride;
    int pos = 0;
    // reverse (util.py:180-184): chunks are walked backwards and every slice is taken from the END of its row with Python's
    // negative indices: index -k resolves to T - k (clamped at 0), and -0 is 0 -- so `x[:-start]` is EMPTY when start == 0 and
    // `x[-first_end:]` is the whole row when first_end == 0, exactly as the reference's expressions evaluate
    auto neg = [T](int k) { return k == 0 ? 0 : max(T - k, 0); };
    for (int step = 0; step < nch; step++) {
        const int ci = reverse ? nch - 1 - step : step;
        int lo, hi;
        if (nch == 1) { lo = 0; hi = T; }
        else if (!reverse) {
            if (ci == 0) { lo = 0; hi = first_end; }
            else if (ci == nch - 1) { lo = start; hi = T; }
            else { lo = start; hi = end; }
        } else {
            if (ci == nch - 1) { lo = 0; hi = neg(start); }
            else if (ci == 0) { lo = neg(first_end); hi = T; }
            else { lo = neg(end); hi = neg(start); }
        }
        lo = max(0, min(lo, T));
        hi = max(lo, min(hi, T));
        const int8_t *row = rows + (size_t)(first + ci) * T;
        for (int base = lo; base < hi; base += 32) {
            int i = base + lane;
            int8_t v = (i < hi) ? row[i] : (int8_t)0;
            unsigned mask = __ballot_sync(0xffffffffu, v != 0);
            if (v != 0) {
                int p = pos + __popc(mask & ((1u << lane) - 1));
                if (p < out_stride) o[p] = v;
            }
            pos += __popc(mask);
        }
    }
    if (lane == 0) out_len[r] = min(pos, out_stride);
}

// posteriors(scores, Max) = one-hot at the arg-max edge of every (t, n): zero the row, set one element
__global__ void onehot_edges_kernel(const int32_t *__restrict__ edges_nt, int T, int N, int S, float *__restrict__ post) {
    const int t = blockIdx.x, n = blockIdx.y;
    float *row = post + ((size_t)t * N + n) * S;
    const int e = edges_nt[(size_t)n * T + t];
    for (int i = threadIdx.x; i < S; i += blockDim.x) row[i] = (i == e) ? 1.0f : 0.0f;
}

// ---- chunk gather ------------------------------------------------------------------------------------
// util.chunk (bonito/util.py:152-166) for a whole read set on the device: chunk c of the batch is samples
// [start, start + L) of read chunk_read[c]; start < 0 means a short read, left-padded with zeros (:160).
template <typename SIG>
__global__ void gather_chunks_kernel(const SIG *__restrict__ signal, const int64_t *__restrict__ read_offset,
                                     const int32_t *__restrict__ read_len, const int32_t *__restrict__ chunk_read,
                                     const int32_t *__restrict__ chunk_start, int L, float *__restrict__ out) {
    const int c = blockIdx.y;
    const int r = chunk_read[c], start = chunk_start[c], len = read_len[r];
    const SIG *src = signal + read_offset[r];
    float *dst = out + (size_t)c * L;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) {
        const int p = start + i;
        dst[i] = (p >= 0 && p < len) ? (float)src[p] : 0.0f;
    }
}

// ---- CTC-CRF loss -----------------------------------------------------------------------------------
__device__ __forceinline__ float logaddexp_exact(float a, float b) {
    float m = fmaxf(a, b);
    float s = XB_ADD(xb_expf(XB_SUB(a, m)), xb_expf(XB_SUB(b, m)));
    return XB_ADD(m, xb_logf(s));
}

// grid = N, block = NT (multiple of 32, >= n positions).  dynamic smem: 2*NT floats + row ring
__global__ void ctc_simple_kernel(const float *__restrict__ scores, int T, int N, int S, const int32_t *__restrict__ targets,
                                  int Lmax, const int32_t *__restrict__ lengths, const float *__restrict__ logz,
                                  int normalise, int n_base, int state_len, float *__restrict__ loss) {
    extern __shared__ __align__(16) float sm[];
    const int NT = blockDim.x, j = threadIdx.x, n = blockIdx.x;
    float *a = sm;                   // 2 * NT
    float *rowbuf = sm + 2 * NT;     // 2 * S  (double buffered score row)
    const int npos = Lmax - (state_len - 1);
    const int NZ = n_base + 1;
    const int32_t *tg = targets + (size_t)n * Lmax;
    const bool act = j < npos;
    // stay edge of position j, and the move edge ENTERING position j (move_indices[j-1] of
    // crf/model.py:113 = stay_indices[j] + targets[j-1] + 1)
    int stay_idx = 0, move_in = 0;
    if (act) {
        int st = 0;
        for (int i = 0; i < state_len; i++) st = st * n_base + max(tg[j + i] - 1, 0);
        stay_idx = st * NZ;
        if (j > 0) move_in = stay_idx + max(tg[j - 1] - 1, 0) + 1;
    }
    const float shift = normalise ? logz[n] / (float)T : 0.0f;
    a[j] = (j == 0) ? 0.0f : XB_NEG_BIG;
    const float *base = scores + (size_t)n * S;
    const size_t row = (size_t)N * S;
    for (int i = j; i < S; i += NT) rowbuf[i] = base[i];
    __syncthreads();
    for (int t = 0; t < T; t++) {
        const float *M = rowbuf + (t & 1) * S;
        float *Mn = rowbuf + ((t + 1) & 1) * S;
        if (t + 1 < T)
            for (int i = j; i < S; i += NT) Mn[i] = base[(size_t)(t + 1) * row + i];
        const float *ac = a + (t & 1) * NT;
        float *an = a + ((t + 1) & 1) * NT;
        if (act) {
            float v = XB_ADD(XB_SUB(M[stay_idx], shift), ac[j]);
            if (j > 0) v = logaddexp_exact(v, XB_ADD(XB_SUB(M[move_in], shift), ac[j - 1]));
            an[j] = v;
        } else {
            an[j] = XB_NEG_BIG;
        }
        __syncthreads();
    }
    if (j == 0) {
        const int len = lengths[n];
        const int last = len + 1 - state_len - 1;
        float z = (last >= 0 && last < npos) ? a[(T & 1) * NT + last] : XB_NEG_BIG;
        loss[n] = -z / (float)len;
    }
}

// Gradient of the per-sequence loss w.r.t. the scores (what autograd gives the reference through seqdist's Logspace
// backward, crf/model.py:118-131):  d loss_n / d scores[t,n,e] = (P_den[t,n,e] - P_num[t,n,e]) / len_n, where P_den are
// the edge posteriors of the full lattice (present only because normalise subtracts logZ/T from every score; the caller
// has put them into `grad`) and P_num the posteriors of the target's stay / move edges under the alignment lattice.
// Forward pass stores alpha (T+1, N, npos), the backward pass walks beta and scatters through a shared-memory row.
__global__ void ctc_simple_bwd_kernel(const float *__restrict__ scores, int T, int N, int S, const int32_t *__restrict__ targets,
                                      int Lmax, const int32_t *__restrict__ lengths, const float *__restrict__ logz,
                                      int normalise, int n_base, int state_len, const float *__restrict__ grad_loss,
                                      float *__restrict__ alpha_ws, float *__restrict__ grad) {
    extern __shared__ __align__(16) float sm[];
    const int NT = blockDim.x, j = threadIdx.x, n = blockIdx.x;
    float *a = sm;                                   // 2 * NT (alpha, then beta)
    int *mv = reinterpret_cast<int *>(sm + 2 * NT);  // NT + 1: move edge entering position j
    float *acc = sm + 3 * NT + 1;                    // S
    float *rowbuf = acc + S;                         // S
    const int npos = Lmax - (state_len - 1);
    const int NZ = n_base + 1;
    const int32_t *tg = targets + (size_t)n * Lmax;
    const bool act = j < npos;
    int stay_idx = 0, move_in = 0;
    if (act) {
        int st = 0;
        for (int i = 0; i < state_len; i++) st = st * n_base + max(tg[j + i] - 1, 0);
        stay_idx = st * NZ;
        if (j > 0) move_in = stay_idx + max(tg[j - 1] - 1, 0) + 1;
    }
    mv[j] = move_in;
    if (j == 0) mv[NT] = 0;
    const float shift = normalise ? logz[n] / (float)T : 0.0f;
    const float *base = scores + (size_t)n * S;
    const size_t row = (size_t)N * S, arow = (size_t)N * npos;
    float *aw = alpha_ws + (size_t)n * npos;
    a[j] = (j == 0) ? 0.0f : XB_NEG_BIG;
    if (act) aw[j] = a[j];
    // Every global read of a step (score row, stored alpha, incoming gradient row) is issued one step ahead into registers,
    // so the three L2 / HBM round trips of a step overlap the previous step's arithmetic instead of following each other.
    constexpr int RPT = 4;                           // row elements per thread: S <= RPT * NT is checked by the launcher
    float rpre[RPT];
    auto fetch_row = [&](int t) {
#pragma unroll
        for (int k = 0; k < RPT; k++) {
            const int e = j + k * NT;
            rpre[k] = (e < S) ? base[(size_t)t * row + e] : 0.0f;
        }
    };
    fetch_row(0);
    __syncthreads();
    for (int t = 0; t < T; t++) {
#pragma unroll
        for (int k = 0; k < RPT; k++)
            if (j + k * NT < S) rowbuf[j + k * NT] = rpre[k];
        __syncthreads();
        if (t + 1 < T) fetch_row(t + 1);
        const float *ac = a + (t & 1) * NT;
        float *an = a + ((t + 1) & 1) * NT;
        float v = XB_NEG_BIG;
        if (act) {
            v = XB_ADD(XB_SUB(rowbuf[stay_idx], shift), ac[j]);
            if (j > 0) v = logaddexp_exact(v, XB_ADD(XB_SUB(rowbuf[move_in], shift), ac[j - 1]));
            aw[(size_t)(t + 1) * arow + j] = v;
        }
        an[j] = v;
        __syncthreads();
    }
    const int len = lengths[n];
    const int last = len + 1 - state_len - 1;
    const bool feasible = last >= 0 && last < npos && a[(T & 1) * NT + last] > -1e37f;
    const float lz = feasible ? a[(T & 1) * NT + last] : 0.0f;
    const float scale = grad_loss[n] / (float)len;
    __syncthreads();
    a[j] = (j == last) ? 0.0f : XB_NEG_BIG;           // beta_T in buffer 0
    float gpre[RPT], at_pre = 0.0f, am1_pre = 0.0f;
    auto fetch_step = [&](int t) {
        fetch_row(t);
        if (normalise) {
            const float *g = grad + ((size_t)t * N + n) * S;
#pragma unroll
            for (int k = 0; k < RPT; k++) {
                const int e = j + k * NT;
                gpre[k] = (e < S) ? g[e] : 0.0f;
            }
        }
        if (act) {
            at_pre = aw[(size_t)t * arow + j];
            if (j > 0) am1_pre = aw[(size_t)t * arow + j - 1];
        }
    };
#pragma unroll
    for (int k = 0; k < RPT; k++) gpre[k] = 0.0f;
    fetch_step(T - 1);
    for (int i = 0; i < T; i++) {
        const int t = T - 1 - i;
        float gcur[RPT];
#pragma unroll
        for (int k = 0; k < RPT; k++) {
            const int e = j + k * NT;
            if (e < S) { rowbuf[e] = rpre[k]; acc[e] = 0.0f; }
            gcur[k] = gpre[k];
        }
        const float at = at_pre, am1 = am1_pre;
        __syncthreads();
        if (t > 0) fetch_step(t - 1);
        const float *b1 = a + (i & 1) * NT;
        float *b0 = a + ((i + 1) & 1) * NT;
        float bnew = XB_NEG_BIG;
        if (act) {
            const float stay_term = XB_ADD(XB_SUB(rowbuf[stay_idx], shift), b1[j]);
            if (feasible) {
                atomicAdd(&acc[stay_idx], xb_expf(XB_SUB(XB_ADD(at, stay_term), lz)));
                if (j > 0) {
                    const float mterm = XB_ADD(XB_SUB(rowbuf[move_in], shift), b1[j]);
                    atomicAdd(&acc[move_in], xb_expf(XB_SUB(XB_ADD(am1, mterm), lz)));
                }
            }
            bnew = stay_term;
            if (j + 1 < npos) bnew = logaddexp_exact(bnew, XB_ADD(XB_SUB(rowbuf[mv[j + 1]], shift), b1[j + 1]));
        }
        b0[j] = bnew;
        __syncthreads();
        float *g = grad + ((size_t)t * N + n) * S;
#pragma unroll
        for (int k = 0; k < RPT; k++) {
            const int e = j + k * NT;
            if (e < S) g[e] = scale * (gcur[k] - acc[e]);
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" {

int xb_stitch(xb_handle *h, const int8_t *rows, int T, const int32_t *chunk_first, const int32_t *chunk_count,
              const int32_t *read_len, int n_reads, int chunksize, int overlap, int stride, int reverse, int8_t *out,
              int out_stride, int32_t *out_len, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, rows && chunk_first && chunk_count && read_len && out && out_len, "NULL buffer");
    XB_CUDA(h, cudaSetDevice(h->device));
    XB_REQUIRE(h, n_reads > 0 && chunksize > overlap && stride > 0, "bad stitch arguments");
    const int warps = 4;
    stitch_kernel<<<(n_reads + warps - 1) / warps, warps * 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        rows, T, chunk_first, chunk_count, read_len, n_reads, chunksize, overlap, stride, reverse, out, out_stride, out_len);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

int xb_gather_chunks(xb_handle *h, const void *signal, int sig_dtype, const int64_t *read_offset, const int32_t *read_len,
                     const int32_t *chunk_read, const int32_t *chunk_start, int n_chunks, int L, float *out, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, signal && read_offset && read_len && chunk_read && chunk_start && out, "NULL buffer");
    XB_CUDA(h, cudaSetDevice(h->device));
    XB_REQUIRE(h, n_chunks > 0 && L > 0, "bad gather arguments");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid((L + 1023) / 1024, n_chunks);
    if (sig_dtype == XB_SIG_F32)
        gather_chunks_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float *>(signal), read_offset, read_len,
                                                         chunk_read, chunk_start, L, out);
    else if (sig_dtype == XB_SIG_I16)
        gather_chunks_kernel<int16_t><<<grid, 256, 0, s>>>(reinterpret_cast<const int16_t *>(signal), read_offset, read_len,
                                                           chunk_read, chunk_start, L, out);
    else
        return xb_fail(h, XB_ERR_ARG, "gather supports fp32 and int16 signal");
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

}  // extern "C"

int xb_onehot_edges(xb_handle *h, const int32_t *edges_nt, int T, int N, int S, float *post, cudaStream_t s) {
    onehot_edges_kernel<<<dim3(T, N), 256, 0, s>>>(edges_nt, T, N, S, post);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

int xb_ctc_loss_impl(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                     const int32_t *lengths, int normalise, float *loss, cudaStream_t s) {
    const int npos = Lmax - (h->state_len - 1);
    XB_REQUIRE(h, npos >= 1 && npos <= 1024, "Lmax=%d unsupported (1 <= Lmax-state_len+1 <= 1024)", Lmax);
    if (normalise)
        if (int rc = xb_decode_alpha(h, scores, T, N, nullptr, h->logz, 0, s)) return rc;
    const int NT = ((npos + 31) / 32) * 32;
    const int S = h->C * h->NZ;
    size_t smem = sizeof(float) * (2 * NT + 2 * S);
    ctc_simple_kernel<<<N, NT, smem, s>>>(scores, T, N, S, targets, Lmax, lengths, h->logz, normalise, h->n_base,
                                         h->state_len, loss);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

// Every argument is checked before the first launch, so a refused call leaves `grad` and the handle's logZ untouched.
int xb_ctc_loss_bwd_impl(xb_handle *h, const float *scores, int T, int N, const int32_t *targets, int Lmax,
                         const int32_t *lengths, int normalise, const float *grad_loss, float *alpha_ws, float *grad,
                         cudaStream_t s) {
    const int npos = Lmax - (h->state_len - 1);
    XB_REQUIRE(h, npos >= 1 && npos <= 1024, "Lmax=%d unsupported (1 <= Lmax-state_len+1 <= 1024)", Lmax);
    const int S = h->C * h->NZ;
    int NT = ((npos + 31) / 32) * 32;
    if (NT * 4 < S) NT = ((S + 127) / 128) * 32;      // the kernel keeps a score row in four registers per thread
    XB_REQUIRE(h, NT <= 1024, "score rows of %d elements are not supported by the loss backward", S);
    if (normalise) {       // logZ (for the shift) and the posteriors of the full lattice, straight into grad
        if (int rc = xb_decode_lin(h, scores, 0, T, N, nullptr, nullptr, nullptr, nullptr, grad, s)) return rc;
        if (int rc = xb_decode_alpha(h, scores, T, N, nullptr, h->logz, 0, s)) return rc;
    }
    size_t smem = sizeof(float) * (3 * NT + 1 + 2 * S);
    if (int rc = xb_smem_attr(h, ctc_simple_bwd_kernel, smem)) return rc;
    ctc_simple_bwd_kernel<<<N, NT, smem, s>>>(scores, T, N, S, targets, Lmax, lengths, h->logz, normalise, h->n_base,
                                             h->state_len, grad_loss, alpha_ws, grad);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
