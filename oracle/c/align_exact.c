/* Plain-C checker of csrc/align.cu (xb_align_counts): local alignment counts written the other way round from the
 * kernel -- full H / D / I matrices, then an explicit traceback with the same preferences.  TEST INFRASTRUCTURE ONLY.
 *
 * The contract (the reference's parasail.sw_trace_striped_32(seq, ref, 8, 4, dnafull), bonito/util.py:402-424, with
 * every letter scored alike):
 *   query row i (seq), reference column j (ref); identical bytes +5, different bytes -4; a gap of length k costs
 *   8 + 4 (k - 1).
 *   D[i][j] = max(H[i][j-1] - 8, D[i][j-1] - 4)   a del column (reference base missing from seq)
 *   I[i][j] = max(H[i-1][j] - 8, I[i-1][j] - 4)   an ins column
 *   H[i][j] = max(0, H[i-1][j-1] +5/-4, D[i][j], I[i][j]);  H = 0 on row 0 and column 0, D / I = -inf there.
 *   Ties: a gap state prefers opening to extending; H prefers the diagonal, then D, then I; the end cell is the highest
 *   H, the first in (i, j) lexicographic order; the traceback stops at an H cell of value 0.  An end score of 0 is the
 *   empty alignment.
 * Output per pair: (score, eq, x, ins, del). */
#include <stdint.h>
#include <stdlib.h>

#define XBO_NEG (-(1 << 28))
#define XBO_MAX_LEN 32767

static int align_one(const int8_t *q, int n, const int8_t *r, int m, int32_t *out) {
    out[0] = out[1] = out[2] = out[3] = out[4] = 0;
    if (n == 0 || m == 0) return 0;
    const size_t W = (size_t)m + 1, cells = ((size_t)n + 1) * W;
    int32_t *H = malloc(cells * sizeof(int32_t)), *D = malloc(cells * sizeof(int32_t)), *I = malloc(cells * sizeof(int32_t));
    if (!H || !D || !I) {
        free(H); free(D); free(I);
        return -1;
    }
    for (size_t j = 0; j < W; j++) { H[j] = 0; D[j] = I[j] = XBO_NEG; }
    int best = 0, bi = 0, bj = 0;
    for (int i = 1; i <= n; i++) {
        int32_t *h = H + (size_t)i * W, *d = D + (size_t)i * W, *in = I + (size_t)i * W;
        const int32_t *hu = h - W, *iu = in - W;
        h[0] = 0; d[0] = in[0] = XBO_NEG;
        for (int j = 1; j <= m; j++) {
            const int dopen = h[j - 1] - 8, dext = d[j - 1] - 4;
            d[j] = dopen >= dext ? dopen : dext;
            const int iopen = hu[j] - 8, iext = iu[j] - 4;
            in[j] = iopen >= iext ? iopen : iext;
            int v = hu[j - 1] + (q[i - 1] == r[j - 1] ? 5 : -4);
            if (d[j] > v) v = d[j];
            if (in[j] > v) v = in[j];
            h[j] = v > 0 ? v : 0;
            if (h[j] > best) { best = h[j]; bi = i; bj = j; }
        }
    }
    int32_t eq = 0, x = 0, ins = 0, del = 0;
    int i = bi, j = bj, state = 0;           /* 0 = H, 1 = D, 2 = I */
    while (best > 0) {
        const size_t at = (size_t)i * W + j;
        if (state == 0) {
            if (H[at] == 0) break;
            const int match = q[i - 1] == r[j - 1];
            if (H[at] == H[at - W - 1] + (match ? 5 : -4)) {
                if (match) eq++; else x++;
                i--; j--;
            } else if (H[at] == D[at]) {
                state = 1;
            } else {
                state = 2;
            }
        } else if (state == 1) {
            del++;
            if (D[at] == H[at - 1] - 8) state = 0;
            j--;
        } else {
            ins++;
            if (I[at] == H[at - W] - 8) state = 0;
            i--;
        }
    }
    free(H); free(D); free(I);
    out[0] = best; out[1] = eq; out[2] = x; out[3] = ins; out[4] = del;
    return 0;
}

/* Pairs [lo, hi) of a batch laid out as for xb_align_counts (host memory); counts (n_pairs, 5).  Returns 0, -1 on a
 * length outside [0, 32767] or beyond its row stride, -2 when memory runs out. */
int xbo_align_counts_range(const int8_t *seq, int seq_stride, const int32_t *seq_len, const int8_t *ref, int ref_stride,
                           const int32_t *ref_len, int lo, int hi, int32_t *counts) {
    for (int p = lo; p < hi; p++) {
        const int n = seq_len[p], m = ref_len[p];
        if (n < 0 || m < 0 || n > XBO_MAX_LEN || m > XBO_MAX_LEN || n > seq_stride || m > ref_stride) return -1;
        if (align_one(seq + (size_t)p * seq_stride, n, ref + (size_t)p * ref_stride, m, counts + (size_t)p * 5)) return -2;
    }
    return 0;
}
