// Batched local alignment for validation accuracy: (score, eq, x, ins, del) of the best local alignment of every
// (decoded sequence, reference) pair, on the device.
//
// Reference: util.accuracy (bonito/util.py:402-424) aligns with parasail.sw_trace_striped_32(seq, ref, 8, 4, dnafull) --
// Smith-Waterman, query = seq, target = ref, a gap of length k costs 8 + 4 (k - 1) -- and counts the columns of the
// alignment's CIGAR.  parasail is not part of this project, so the contract is written down here and checked against
// oracle/c/align_exact.c (full matrices + explicit traceback), integer for integer:
//   scoring   identical letters +5, different letters -4, for every byte value.  dnafull agrees on A/C/G/T; it reads Y as
//             the IUPAC pyrimidine and has no X, whereas here X and Y are ordinary letters.
//   recurrences (query row i, reference column j; every state carries the counts (eq, x, ins, del) of the path it ends)
//             D[i][j] = max(H[i][j-1] - 8, D[i][j-1] - 4)       + one del column (a reference base missing from seq)
//             I[i][j] = max(H[i-1][j] - 8, I[i-1][j] - 4)       + one ins column
//             H[i][j] = max(0, H[i-1][j-1] +5/-4, D[i][j], I[i][j])
//   ties      in a gap state opening wins over extending; in H the order is diagonal, then D, then I; a best candidate
//             <= 0 restarts H at 0 with zero counts; the end cell is the highest H, the first in (i, j) lexicographic
//             order; an end score of 0 is the empty alignment (all counts 0).
// Carrying the counts forward with these preferences yields exactly the path a traceback with the same preferences
// walks, so no traceback matrix is kept.  Under these rules an optimal local alignment starts and ends with a match
// column, so the clipping in the reference's parasail_to_sam (a leading I becomes a soft clip, a leading D is dropped)
// never applies: the counts are the CIGAR's.
//
// Layout: one warp per pair, WARPS pairs per CTA.  Lane k owns B consecutive reference columns of a band of 32 * B
// columns and keeps their H and I states (with counts) of the previous query row in registers.  The warp runs a skewed
// wavefront over the query rows: at step s lane k works on row s - k + 1, taking the H / D values (and the query letter)
// of its left neighbour's last column for that row by __shfl_up_sync.  References longer than a band are processed band
// after band; the right-edge column of a band goes to a global workspace that lane 0 reads in the next band.
// Counts are packed two per 32-bit word (eq | x << 16, ins | del << 16): lengths <= 32767 keep every field below 2^16.
// Integer work only; the bound is integer issue along the wavefront's dependency chain.
#include "xb_common.cuh"

namespace {

constexpr int B = 16;                   // reference columns per lane
constexpr int BAND = 32 * B;            // reference columns per band
constexpr int WARPS = 4;                // pairs per CTA
constexpr int MAX_LEN = 32767;
constexpr int NEG = -(1 << 28);         // minus infinity of the gap states (no overflow after 2^15 extensions)
constexpr uint32_t C_EQ = 1u, C_X = 1u << 16, C_INS = 1u, C_DEL = 1u << 16;

struct Best {
    int s, i, j;
    uint32_t lo, hi;
};

__device__ __forceinline__ bool better(const Best &a, const Best &b) {
    return a.s > b.s || (a.s == b.s && (a.i < b.i || (a.i == b.i && a.j < b.j)));
}

__device__ __forceinline__ int sel(bool p, int a, int b) { return p ? a : b; }
__device__ __forceinline__ uint32_t sel(bool p, uint32_t a, uint32_t b) { return p ? a : b; }

// edge: per pair 2 buffers x edge_rows rows x 2 int4 = {H, H lo, H hi, D}, {D lo, D hi, -, -} of a band's last column
__global__ void __launch_bounds__(32 * WARPS)
align_counts_kernel(const int8_t *__restrict__ seq, int seq_stride, const int32_t *__restrict__ seq_len,
                    const int8_t *__restrict__ ref, int ref_stride, const int32_t *__restrict__ ref_len, int n_pairs,
                    int32_t *__restrict__ counts, int4 *__restrict__ edge, int edge_rows) {
    const int lane = threadIdx.x & 31;
    const int pair = blockIdx.x * WARPS + (threadIdx.x >> 5);
    if (pair >= n_pairs) return;                         // warp-uniform: no block-level barrier follows
    const int n = seq_len[pair], m = ref_len[pair];
    const int8_t *q = seq + (size_t)pair * seq_stride;
    const int8_t *r = ref + (size_t)pair * ref_stride;
    const int bands = n > 0 ? (m + BAND - 1) / BAND : 0;
    Best best = {0, 0, 0, 0u, 0u};                       // warp-uniform running best over the bands

    for (int band = 0; band < bands; ++band) {
        const int j0 = band * BAND + lane * B;           // this lane's columns are j0 + 1 .. j0 + B (1-based)
        const int nvalid = min(max(m - j0, 0), B);
        int rl[B], hs[B], is[B];
        uint32_t hlo[B], hhi[B], ilo[B], ihi[B];
#pragma unroll
        for (int c = 0; c < B; ++c) {
            rl[c] = c < nvalid ? (int)r[j0 + c] : 0x100;  // never equal to a query byte
            hs[c] = 0; hlo[c] = 0u; hhi[c] = 0u;          // row 0: H = 0, I = -inf
            is[c] = NEG; ilo[c] = 0u; ihi[c] = 0u;
        }
        const int4 *ein = edge + (size_t)pair * 4 * edge_rows + (size_t)((band + 1) & 1) * 2 * edge_rows;
        int4 *eout = edge + (size_t)pair * 4 * edge_rows + (size_t)(band & 1) * 2 * edge_rows;
        const bool store_edge = lane == 31 && band + 1 < bands;
        // lane 0's left column: the boundary (band 0) or the previous band's edge, prefetched one row ahead
        int pq = lane == 0 ? (int)q[0] : 0;
        int4 pe0 = make_int4(0, 0, 0, NEG), pe1 = make_int4(0, 0, 0, 0);
        if (lane == 0 && band > 0) { pe0 = ein[0]; pe1 = ein[1]; }
        int dg_h = 0;                                    // H[i-1][j0] of the row this lane works on next
        uint32_t dg_lo = 0u, dg_hi = 0u;
        int oh = 0, od = NEG, oq = 0;                    // what the right neighbour takes at the next step
        uint32_t ohlo = 0u, ohhi = 0u, odlo = 0u, odhi = 0u;
        Best lb = {0, 0, 0, 0u, 0u};
        for (int s = 0; s < n + 31; ++s) {
            int lh = __shfl_up_sync(0xffffffffu, oh, 1);
            uint32_t lhlo = __shfl_up_sync(0xffffffffu, ohlo, 1), lhhi = __shfl_up_sync(0xffffffffu, ohhi, 1);
            int ld = __shfl_up_sync(0xffffffffu, od, 1);
            uint32_t ldlo = __shfl_up_sync(0xffffffffu, odlo, 1), ldhi = __shfl_up_sync(0xffffffffu, odhi, 1);
            int lq = __shfl_up_sync(0xffffffffu, oq, 1);
            if (lane == 0) {
                lq = pq; lh = pe0.x; lhlo = (uint32_t)pe0.y; lhhi = (uint32_t)pe0.z; ld = pe0.w;
                ldlo = (uint32_t)pe1.x; ldhi = (uint32_t)pe1.y;
                if (s + 1 < n) {
                    pq = q[s + 1];
                    if (band > 0) { pe0 = ein[2 * (s + 1)]; pe1 = ein[2 * (s + 1) + 1]; }
                }
            }
            const int i = s - lane + 1;
            if (i >= 1 && i <= n) {
                int left_h = lh, left_d = ld;
                uint32_t left_lo = lhlo, left_hi = lhhi, left_dlo = ldlo, left_dhi = ldhi;
                int d_h = dg_h;
                uint32_t d_lo = dg_lo, d_hi = dg_hi;
#pragma unroll
                for (int c = 0; c < B; ++c) {
                    const int dopen = left_h - 8, dext = left_d - 4;
                    const bool dto = dopen >= dext;
                    const int dv = sel(dto, dopen, dext);
                    const uint32_t dlo = sel(dto, left_lo, left_dlo), dhi = sel(dto, left_hi, left_dhi) + C_DEL;
                    const int iopen = hs[c] - 8, iext = is[c] - 4;
                    const bool ito = iopen >= iext;
                    const int iv = sel(ito, iopen, iext);
                    const uint32_t nilo = sel(ito, hlo[c], ilo[c]), nihi = sel(ito, hhi[c], ihi[c]) + C_INS;
                    const bool eq = lq == rl[c];
                    int h = d_h + (eq ? 5 : -4);
                    uint32_t clo = d_lo + (eq ? C_EQ : C_X), chi = d_hi;
                    if (dv > h) { h = dv; clo = dlo; chi = dhi; }
                    if (iv > h) { h = iv; clo = nilo; chi = nihi; }
                    if (h <= 0) { h = 0; clo = 0u; chi = 0u; }
                    d_h = hs[c]; d_lo = hlo[c]; d_hi = hhi[c];
                    hs[c] = h; hlo[c] = clo; hhi[c] = chi;
                    is[c] = iv; ilo[c] = nilo; ihi[c] = nihi;
                    left_h = h; left_lo = clo; left_hi = chi;
                    left_d = dv; left_dlo = dlo; left_dhi = dhi;
                    if (h > lb.s && c < nvalid) { lb.s = h; lb.i = i; lb.j = j0 + c + 1; lb.lo = clo; lb.hi = chi; }
                }
                dg_h = lh; dg_lo = lhlo; dg_hi = lhhi;
                oh = left_h; ohlo = left_lo; ohhi = left_hi; od = left_d; odlo = left_dlo; odhi = left_dhi; oq = lq;
                if (store_edge) {
                    eout[2 * (i - 1)] = make_int4(left_h, (int)left_lo, (int)left_hi, left_d);
                    eout[2 * (i - 1) + 1] = make_int4((int)left_dlo, (int)left_dhi, 0, 0);
                }
            }
        }
        // the band's best cell: highest score, then first in (i, j) order
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            Best o;
            o.s = __shfl_xor_sync(0xffffffffu, lb.s, off);
            o.i = __shfl_xor_sync(0xffffffffu, lb.i, off);
            o.j = __shfl_xor_sync(0xffffffffu, lb.j, off);
            o.lo = __shfl_xor_sync(0xffffffffu, lb.lo, off);
            o.hi = __shfl_xor_sync(0xffffffffu, lb.hi, off);
            if (better(o, lb)) lb = o;
        }
        if (better(lb, best)) best = lb;
        __syncwarp();                                    // the edge written by lane 31 is read by lane 0 next band
    }
    if (lane == 0) {
        int32_t *o = counts + (size_t)pair * 5;
        o[0] = best.s;
        o[1] = (int32_t)(best.lo & 0xffffu);
        o[2] = (int32_t)(best.lo >> 16);
        o[3] = (int32_t)(best.hi & 0xffffu);
        o[4] = (int32_t)(best.hi >> 16);
    }
}

}  // namespace

extern "C" {

int xb_align_counts(const int8_t *seq, int seq_stride, const int32_t *seq_len, const int8_t *ref, int ref_stride,
                    const int32_t *ref_len, int n_pairs, int32_t *counts, void *stream) {
    if (!seq || !seq_len || !ref || !ref_len || !counts || n_pairs < 0 || seq_stride < 0 || ref_stride < 0)
        return xb_fail(nullptr, XB_ERR_ARG, "xb_align_counts: bad arguments");
    if (n_pairs == 0) return XB_OK;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    // the lengths are validated on the host and size the band workspace
    std::vector<int32_t> lens(2 * (size_t)n_pairs);
    cudaError_t e = cudaMemcpyAsync(lens.data(), seq_len, sizeof(int32_t) * n_pairs, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(lens.data() + n_pairs, ref_len, sizeof(int32_t) * n_pairs, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return xb_fail(nullptr, XB_ERR_CUDA, "xb_align_counts: reading the lengths failed: %s", cudaGetErrorString(e));
    int max_n = 0, max_m = 0;
    for (int p = 0; p < n_pairs; ++p) {
        const int n = lens[p], m = lens[n_pairs + p];
        if (n < 0 || m < 0 || n > MAX_LEN || m > MAX_LEN)
            return xb_fail(nullptr, XB_ERR_ARG, "xb_align_counts: pair %d has lengths %d / %d outside [0, %d]", p, n, m, MAX_LEN);
        if (n > seq_stride || m > ref_stride)
            return xb_fail(nullptr, XB_ERR_ARG, "xb_align_counts: pair %d has lengths %d / %d beyond the row strides %d / %d",
                           p, n, m, seq_stride, ref_stride);
        max_n = n > max_n ? n : max_n;
        max_m = m > max_m ? m : max_m;
    }
    int4 *edge = nullptr;
    if (max_m > BAND && max_n > 0) {
        e = cudaMallocAsync(reinterpret_cast<void **>(&edge), (size_t)n_pairs * 4 * max_n * sizeof(int4), s);
        if (e != cudaSuccess) return xb_fail(nullptr, XB_ERR_NOMEM, "xb_align_counts: workspace: %s", cudaGetErrorString(e));
    }
    align_counts_kernel<<<(n_pairs + WARPS - 1) / WARPS, 32 * WARPS, 0, s>>>(seq, seq_stride, seq_len, ref, ref_stride,
                                                                           ref_len, n_pairs, counts, edge, max_n);
    e = cudaGetLastError();
    if (edge) cudaFreeAsync(edge, s);
    if (e != cudaSuccess) return xb_fail(nullptr, XB_ERR_CUDA, "xb_align_counts: launch failed: %s", cudaGetErrorString(e));
    return XB_OK;
}

}  // extern "C"
