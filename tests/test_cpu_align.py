"""The local alignment contract of validation accuracy (csrc/align.cu, oracle/c/align_exact.c) on the host: the C checker
against known answers, an independent pure-Python DP that records its choices and walks them back, and a brute-force
enumeration of every local alignment of short strings; plus the host halves of util.accuracy (decode_ref, the accuracy
expressions on counts)."""
import numpy as np
import pytest
import torch

from oracle import align_exact
from xna_basecaller_b200 import util

# seq, ref -> (score, eq, x, ins, del), accuracy at min_coverage 0.5, at 0, balanced
KNOWN = [
    ('ACGTACGT', 'ACGTACGT', (40, 8, 0, 0, 0), 100.0, 100.0, 100.0),
    ('ACGTTACGT', 'ACGTACGT', (32, 8, 0, 1, 0), 800 / 9, 800 / 9, 87.5),
    ('ACGACGTA', 'ACGTACGTA', (32, 8, 0, 0, 1), 800 / 9, 800 / 9, 800 / 9),
    ('AXGTACGT', 'ACGTACGT', (31, 7, 1, 0, 0), 87.5, 87.5, 87.5),
    ('ACGTACGTAAAAAAAA', 'ACGTACGTCCCCCCCCCC', (40, 8, 0, 0, 0), 0.0, 100.0, 100.0),
    ('TTTT', 'GGGG', (0, 0, 0, 0, 0), 0.0, 0.0, 0.0),
]


def test_checker_known_answers():
    got = align_exact.align_strings([k[0] for k in KNOWN], [k[1] for k in KNOWN])
    for (seq, ref, want, acc_half, acc_zero, acc_bal), row in zip(KNOWN, got):
        assert tuple(row) == want, (seq, ref, row)
        assert util._accuracy(row, len(ref), False, 0.5) == pytest.approx(acc_half, abs=1e-12)
        assert util._accuracy(row, len(ref), False, 0.0) == pytest.approx(acc_zero, abs=1e-12)
        assert util._accuracy(row, len(ref), True, 0.0) == pytest.approx(acc_bal, abs=1e-12)


def _python_dp(q, r):
    """Smith-Waterman with affine gaps (open 8, extend 4; +5 / -4), written with explicit back-pointers: every cell
    records which candidate it took under the tie rules, and the path is walked back from the first highest H."""
    n, m = len(q), len(r)
    NEG = -10 ** 9
    H = [[0] * (m + 1) for _ in range(n + 1)]
    D = [[NEG] * (m + 1) for _ in range(n + 1)]
    I = [[NEG] * (m + 1) for _ in range(n + 1)]
    pH = [[None] * (m + 1) for _ in range(n + 1)]      # 'M' diagonal, 'D', 'I', None = start
    pD = [[None] * (m + 1) for _ in range(n + 1)]      # True = opened from H
    pI = [[None] * (m + 1) for _ in range(n + 1)]
    best, end = 0, None
    for i in range(1, n + 1):
        for j in range(1, m + 1):
            o, e = H[i][j - 1] - 8, D[i][j - 1] - 4
            D[i][j], pD[i][j] = (o, True) if o >= e else (e, False)
            o, e = H[i - 1][j] - 8, I[i - 1][j] - 4
            I[i][j], pI[i][j] = (o, True) if o >= e else (e, False)
            cands = [(H[i - 1][j - 1] + (5 if q[i - 1] == r[j - 1] else -4), 'M'), (D[i][j], 'D'), (I[i][j], 'I')]
            v, how = cands[0]
            for c in cands[1:]:
                if c[0] > v:
                    v, how = c
            H[i][j], pH[i][j] = (v, how) if v > 0 else (0, None)
            if H[i][j] > best:
                best, end = H[i][j], (i, j)
    counts = {'=': 0, 'X': 0, 'I': 0, 'D': 0}
    if end is None:
        return (0, 0, 0, 0, 0)
    (i, j), state = end, 'H'
    while True:
        if state == 'H':
            how = pH[i][j]
            if how is None:
                break
            if how == 'M':
                counts['=' if q[i - 1] == r[j - 1] else 'X'] += 1
                i, j = i - 1, j - 1
            else:
                state = how
        elif state == 'D':
            counts['D'] += 1
            state = 'H' if pD[i][j] else 'D'
            j -= 1
        else:
            counts['I'] += 1
            state = 'H' if pI[i][j] else 'I'
            i -= 1
    return (best, counts['='], counts['X'], counts['I'], counts['D'])


def _mutate(rs, s, rate, letters):
    out = []
    for ch in s:
        u = rs.rand()
        if u < rate / 3:
            out.append(letters[rs.randint(len(letters))])
        elif u < 2 * rate / 3:
            out.append(ch)
            out.append(letters[rs.randint(len(letters))])
        elif u >= rate:
            out.append(ch)
    return ''.join(out)


def _pairs(seed, count):
    """Random, mutated (substitutions / insertions / deletions), single-letter runs, no common letter, empty sides."""
    rs = np.random.RandomState(seed)
    abc = 'ACGTXY'
    rnd = lambda n, a=abc: ''.join(a[k] for k in rs.randint(len(a), size=n))
    pairs = []
    for k in range(count):
        kind = k % 6
        if kind == 0:
            pairs.append((rnd(rs.randint(0, 25)), rnd(rs.randint(0, 25))))
        elif kind in (1, 2):
            s = rnd(rs.randint(1, 30))
            pairs.append((_mutate(rs, s, rs.choice([0.1, 0.3, 0.6]), abc), s))
        elif kind == 3:
            a, b = abc[rs.randint(6)], abc[rs.randint(6)]
            pairs.append((a * rs.randint(0, 15) + rnd(rs.randint(0, 3)), b * rs.randint(0, 15)))
        elif kind == 4:
            pairs.append((rnd(rs.randint(0, 20), 'AC'), rnd(rs.randint(0, 20), 'GT')))
        else:
            s = rnd(rs.randint(0, 12))
            pairs.append((s, '') if rs.rand() < 0.5 else ('', s))
    return pairs


def test_checker_matches_python_traceback():
    pairs = _pairs(11, 3000)
    got = align_exact.align_strings([p[0] for p in pairs], [p[1] for p in pairs], threads=4)
    for (q, r), row in zip(pairs, got):
        assert tuple(row) == _python_dp(q, r), (q, r, row)


def _brute_force_score(q, r):
    """Best score over every local alignment: every global alignment of the whole strings (all column sequences), every
    contiguous run of its columns scored on its own (a run is an alignment of two substrings, and every alignment of two
    substrings is such a run), and the empty alignment."""
    best = 0

    def score(cols):
        s, prev = 0, None
        for c in cols:
            if c in 'MX':
                s += 5 if c == 'M' else -4
            else:
                s -= 4 if prev == c else 8
            prev = c
        return s

    def walk(i, j, cols):
        nonlocal best
        if i == len(q) and j == len(r):
            for a in range(len(cols)):
                for b in range(a + 1, len(cols) + 1):
                    best = max(best, score(cols[a:b]))
            return
        if i < len(q) and j < len(r):
            walk(i + 1, j + 1, cols + ('M' if q[i] == r[j] else 'X'))
        if i < len(q):
            walk(i + 1, j, cols + 'I')
        if j < len(r):
            walk(i, j + 1, cols + 'D')

    walk(0, 0, '')
    return best


def test_checker_score_equals_brute_force():
    rs = np.random.RandomState(5)
    pairs = []
    for k in range(150):
        n, m = (rs.randint(0, 6), rs.randint(0, 6)) if k % 10 else (6, 6) if k % 20 else (6, rs.randint(0, 6))
        abc = 'AC' if k % 3 == 0 else 'ACG'
        pairs.append((''.join(rs.choice(list(abc), n)), ''.join(rs.choice(list(abc), m))))
    pairs.append(('AAGAA', 'AAAA'))                    # a gap that pays for itself: 4 * 5 - 8 > 2 * 5
    got = align_exact.align_strings([p[0] for p in pairs], [p[1] for p in pairs])
    for (q, r), row in zip(pairs, got):
        assert row[0] == _brute_force_score(q, r), (q, r, row)


def test_decode_ref():
    labels = ['N', 'A', 'C', 'G', 'T', 'X']
    assert util.decode_ref(torch.tensor([1, 2, 3, 4, 5, 0, 0]), labels) == 'ACGTX'
    assert util.decode_ref(np.array([0, 5, 0, 1]), labels) == 'XA'
    assert util.decode_ref(torch.zeros(4, dtype=torch.int64), labels) == ''


def test_accuracy_expressions_on_counts():
    # coverage counts the alignment's columns, gaps included, against len(ref)
    assert util._accuracy((10, 2, 0, 0, 0), 6, False, 0.5) == 0.0         # 2 / 6 columns: below min_coverage
    assert util._accuracy((10, 2, 0, 0, 0), 6, False, 0.0) == 100.0
    assert util._accuracy((10, 2, 0, 1, 0), 6, False, 0.5) == 2 / 3 * 100     # 3 / 6 is not below 0.5; the reference's order of operations
    assert util._accuracy((10, 2, 0, 1, 0), 6, True, 0.5) == pytest.approx(50.0)
    assert util._accuracy((0, 0, 0, 0, 0), 0, False, 0.0) == 0.0          # empty reference
