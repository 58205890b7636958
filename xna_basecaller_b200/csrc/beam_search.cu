// Beam-search decode over the CTC-CRF lattice for any alphabet size (SURVEY 8f N4).
//
// Reference context: compute_scores' beam branch (bonito/crf/basecall.py:33-46) hands the scores to koi.decode.beam_search
// (koi-cuda102==0.0.5, third-party, closed to alphabets other than ACGT: bonito/util.py:299-313 switches it off for the UB
// models, which therefore only ever decode with Viterbi).  This file gives the UB alphabets the same kind of decoder: a
// beam over (emitted sequence, lattice state) pairs that SUMS the alignments of a sequence (Log semiring) instead of
// following the single best path, guided by the exact backward scores.  koi's source is not part of the reference, so the
// algorithm is restated from the published description of ONT's CRF beam search and pinned by brute force
// (tests: on a lattice small enough for the beam to be exhaustive it returns the most probable label sequence) and
// bit for bit against the plain-C statement in oracle/c/crf_exact.c (xbo_crf_beam_search) -- "parity unpinned" against koi.
//
// Per sequence (one CTA), with beta = Log-semiring backward scores (beta_T = 0):
//   t = 0: the beam holds the W states with the largest beta_0 (ties: lower state), score 0, hash = state + 1
//   step t: every element (hash, s, a) proposes NZ candidates: stay (hash, s, a + M_t[s,0]) and, for j < n_base, the move into
//           s' = (s % n^(L-1)) * n + j through edge k = 1 + s / n^(L-1):  (hash * FNV + j + 1, s', a + M_t[s',k]); the label
//           reported for the move is k (the convention of CTC_CRF.viterbi: 1 + the base dropped from the state;
//           bonito/crf/model.py:92-95), so beam and Viterbi strings are directly comparable;
//           candidates with the same (hash, state) are the same sequence prefix reached by different alignments: the
//           earliest one absorbs the others with logsumexp (ascending candidate order);
//           the surviving candidates are ranked by a + beta_{t+1}[state] (ties: lower candidate index); the best W within
//           beam_cut of the leader form the next beam, stored best first;
//   end:   the leader at t = T is traced back: labels, moves (1 where a base was emitted), and a phred quality per base from
//           the transition probability of its move, exp(M_t[s',k] + beta_{t+1}[s'] - beta_t[s]) (the quantity
//           CTC_CRF.compute_transition_probs normalises, crf/model.py:63-76): q = clamp(round(-10 log10(max(1 - p, 1e-5))), 1, 50).
#include "xb_common.cuh"
#include "xb_exact_math.h"
#include "crf_lattice.cuh"

namespace {

constexpr int BW_MAX = 32;                 // beam width limit (koi's default beam_width)
constexpr int NT_BEAM = 256;               // threads: one per candidate (BW_MAX * NZ <= 224 for n_base <= 6)
constexpr unsigned long long FNV = 1099511628211ULL;

struct BeamArgs {
    const float *scores, *beta;            // (T, N, C*NZ), (T+1, N, C)
    int T, N, C, NZ, n_base, n_pow;        // n_pow = n_base^(state_len-1)
    int beam_width;
    float beam_cut;
    int8_t *seq, *qstring, *moves;         // (N, T) each; qstring / moves may be NULL
    int32_t *lens;
    xbcrf::Alphabet abc;
};

__global__ void __launch_bounds__(NT_BEAM) beam_search_kernel(const BeamArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // beam (double buffered): score, state, hash; candidates: score, rank key, state, hash, first, alive
    float *bscore = reinterpret_cast<float *>(smem_raw);                 // 2 * BW_MAX
    int *bstate = reinterpret_cast<int *>(bscore + 2 * BW_MAX);          // 2 * BW_MAX
    unsigned long long *bhash = reinterpret_cast<unsigned long long *>(bstate + 2 * BW_MAX);   // 2 * BW_MAX
    float *cscore = reinterpret_cast<float *>(bhash + 2 * BW_MAX);       // NT_BEAM
    float *ckey = cscore + NT_BEAM;                                      // NT_BEAM
    int *cstate = reinterpret_cast<int *>(ckey + NT_BEAM);               // NT_BEAM
    int *cfirst = cstate + NT_BEAM;                                      // NT_BEAM
    unsigned long long *chash = reinterpret_cast<unsigned long long *>(cfirst + NT_BEAM);      // NT_BEAM
    int *nbeam = reinterpret_cast<int *>(chash + NT_BEAM);               // 2
    float *rmax = reinterpret_cast<float *>(nbeam + 2);                  // 1 (+1 pad)
    int *istate = reinterpret_cast<int *>(rmax + 2);                     // BW_MAX: states of the initial beam
    unsigned char *back = reinterpret_cast<unsigned char *>(istate + BW_MAX);   // T * BW_MAX: parent | label << 5
    signed char *lab = reinterpret_cast<signed char *>(back + (size_t)a.T * BW_MAX);           // T labels of the winner
    unsigned char *qual = reinterpret_cast<unsigned char *>(lab + a.T);  // T
    const int n = blockIdx.x, i = threadIdx.x;
    const int C = a.C, NZ = a.NZ, W = a.beam_width, T = a.T;
    const size_t S = (size_t)C * NZ;
    const float *beta0 = a.beta + (size_t)n * C;
    const size_t brow = (size_t)a.N * C;

    // ---- t = 0: top-W states by beta_0 (rank by counting; ties -> lower state)
    for (int c = i; c < C; c += NT_BEAM) {
        const float v = beta0[c];
        int rank = 0;
        for (int d = 0; d < C; d++) {
            const float u = beta0[d];
            rank += (u > v) || (u == v && d < c);
        }
        if (rank < W) { bscore[rank] = 0.0f; bstate[rank] = c; istate[rank] = c; bhash[rank] = (unsigned long long)c + 1ULL; }
    }
    if (i == 0) nbeam[0] = min(W, C);
    __syncthreads();

    for (int t = 0; t < T; t++) {
        const int cur = t & 1, nxt = cur ^ 1;
        const int nb = nbeam[cur], ncand = nb * NZ;
        const float *M = a.scores + ((size_t)t * a.N + n) * S;
        const float *b1 = a.beta + (size_t)(t + 1) * brow + (size_t)n * C;
        // 1. candidates
        int e = 0, k = 0;
        if (i < ncand) {
            e = i / NZ; k = i - e * NZ;
            const int s = bstate[cur * BW_MAX + e];
            int s2 = s, edge = s * NZ;
            unsigned long long h = bhash[cur * BW_MAX + e];
            if (k > 0) {
                s2 = (s % a.n_pow) * a.n_base + (k - 1);
                edge = s2 * NZ + 1 + s / a.n_pow;
                h = h * FNV + (unsigned long long)k;
            }
            cscore[i] = XB_ADD(bscore[cur * BW_MAX + e], M[edge]);
            cstate[i] = s2;
            chash[i] = h;
        }
        __syncthreads();
        // 2. merge equal (hash, state): first[i] = lowest index with my key; leaders absorb the rest with logsumexp
        int first = i;
        if (i < ncand) {
            const unsigned long long h = chash[i];
            const int s2 = cstate[i];
            for (int j = 0; j < i; j++)
                if (chash[j] == h && cstate[j] == s2) { first = j; break; }
            cfirst[i] = first;
        }
        __syncthreads();
        float sc = XB_NEG_BIG, key = XB_NEG_BIG;
        bool alive = false;
        if (i < ncand && first == i) {
            float m = cscore[i];
            for (int j = i + 1; j < ncand; j++)
                if (cfirst[j] == i) m = fmaxf(m, cscore[j]);
            float ssum = 0.0f;
            bool any = false;
            for (int j = i; j < ncand; j++)
                if (cfirst[j] == i) {
                    const float ex = xb_expf(XB_SUB(cscore[j], m));
                    ssum = any ? XB_ADD(ssum, ex) : ex;
                    any = true;
                }
            sc = XB_ADD(m, xb_logf(ssum));
            key = XB_ADD(sc, b1[cstate[i]]);
            alive = true;
        }
        __syncthreads();              // every leader has read the raw candidate scores
        if (i < ncand) { cscore[i] = sc; ckey[i] = alive ? key : XB_NEG_BIG; cfirst[i] = alive ? 1 : 0; }
        __syncthreads();
        // 3. rank the leaders by key (descending; ties -> lower index); keep the best W within beam_cut of the best
        int rank = 0;
        float best = XB_NEG_BIG;
        if (i < ncand) {
            for (int j = 0; j < ncand; j++)
                if (cfirst[j]) {
                    const float u = ckey[j];
                    best = fmaxf(best, u);
                    rank += alive && ((u > key) || (u == key && j < i));
                }
        }
        if (i == 0) nbeam[nxt] = 0;
        __syncthreads();
        if (alive && rank < W && key >= XB_SUB(best, a.beam_cut)) {
            bscore[nxt * BW_MAX + rank] = sc;
            bstate[nxt * BW_MAX + rank] = cstate[i];
            bhash[nxt * BW_MAX + rank] = chash[i];
            back[(size_t)t * BW_MAX + rank] = (unsigned char)(e | (k << 5));
            atomicAdd(&nbeam[nxt], 1);           // survivors have ranks 0 .. count-1 (ranks are a permutation of the leaders)
        }
        __syncthreads();
    }
    // ---- trace back the leader (slot 0: largest score + beta_T = score), then walk the path forward for the qualities
    if (i == 0) {
        int slot = 0;
        for (int t = T - 1; t >= 0; t--) {
            const unsigned char bk = back[(size_t)t * BW_MAX + slot];
            lab[t] = (signed char)(bk >> 5);
            slot = bk & 31;
        }
        // walk the path forward: the traceback stored the NEW base (b + 1) of every move; the emitted label follows
        // CTC_CRF.viterbi's convention, the edge index 1 + (base dropped from the source state)
        int s = istate[slot];
        for (int t = 0; t < T; t++) {
            const int b1 = lab[t];
            unsigned char q = 0;
            if (b1 > 0) {
                const int s2 = (s % a.n_pow) * a.n_base + (b1 - 1), k = 1 + s / a.n_pow;
                const float *M = a.scores + ((size_t)t * a.N + n) * S;
                const float lp = XB_SUB(XB_ADD(M[s2 * NZ + k], a.beta[(size_t)(t + 1) * brow + (size_t)n * C + s2]),
                                        a.beta[(size_t)t * brow + (size_t)n * C + s]);
                float err = XB_SUB(1.0f, xb_expf(lp));
                err = err < 1e-5f ? 1e-5f : err;
                const float qf = XB_MUL(-4.34294481903251828f, xb_logf(err));      // -10 log10(err)
                int qi = (int)(XB_ADD(qf, 0.5f));
                qi = qi < 1 ? 1 : (qi > 50 ? 50 : qi);
                q = (unsigned char)(33 + qi);
                lab[t] = (signed char)k;
                s = s2;
            }
            qual[t] = q;
        }
    }
    __syncthreads();
    // ---- outputs: moves, left-packed letters and qualities
    if (a.moves)
        for (int t = i; t < T; t += NT_BEAM) a.moves[(size_t)n * T + t] = lab[t] != 0;
    if (i == 0) {
        int pos = 0;
        for (int t = 0; t < T; t++)
            if (lab[t] != 0) {
                a.seq[(size_t)n * T + pos] = (int8_t)a.abc.ch[(int)lab[t]];
                if (a.qstring) a.qstring[(size_t)n * T + pos] = (int8_t)qual[t];
                pos++;
            }
        for (int p = pos; p < T; p++) {
            a.seq[(size_t)n * T + p] = 0;
            if (a.qstring) a.qstring[(size_t)n * T + p] = 0;
        }
        a.lens[n] = pos;
    }
}

}  // namespace

int xb_beam_search_impl(xb_handle *h, const float *scores, const float *beta, int T, int N, int beam_width, float beam_cut,
                        int8_t *seq, int8_t *qstring, int8_t *moves, int32_t *lens, cudaStream_t s) {
    XB_REQUIRE(h, beam_width >= 1 && beam_width <= BW_MAX, "beam_width must be in 1..%d", BW_MAX);
    XB_REQUIRE(h, beam_width * h->NZ <= NT_BEAM, "beam_width * (n_base + 1) must be <= %d", NT_BEAM);
    BeamArgs a;
    a.scores = scores; a.beta = beta; a.T = T; a.N = N; a.C = h->C; a.NZ = h->NZ; a.n_base = h->n_base;
    a.n_pow = h->C / h->n_base;
    a.beam_width = beam_width; a.beam_cut = beam_cut;
    a.seq = seq; a.qstring = qstring; a.moves = moves; a.lens = lens;
    for (int i = 0; i < 16; i++) a.abc.ch[i] = h->alphabet[i];
    const size_t sm = 2 * BW_MAX * (4 + 4 + 8) + NT_BEAM * (4 + 4 + 4 + 4 + 8) + 16 + BW_MAX * 4 + (size_t)T * BW_MAX + 2 * (size_t)T + 16;
    if (int rc = xb_smem_attr(h, beam_search_kernel, sm)) return rc;
    XB_REQUIRE(h, sm <= 227 * 1024, "T=%d is too long for the beam search's shared-memory traceback", T);
    beam_search_kernel<<<N, NT_BEAM, sm, s>>>(a);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}
