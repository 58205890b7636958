"""ctypes front-end of oracle/c/align_exact.c: the integer-exact checker of the local alignment counts of validation
accuracy (xb_align_counts).  Built on first use, or by build(), into oracle/_build/libxb_align_oracle.so.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, 'c', 'align_exact.c')
_SO = os.path.join(_HERE, '_build', 'libxb_align_oracle.so')
_lib = None


def build(force=False):
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        cc = os.environ.get('CC', 'gcc')
        subprocess.check_call([cc, '-O2', '-fPIC', '-shared', '-std=c11', '-Wall', '-Wextra', '-o', _SO, _SRC])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_SO)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def align_counts(seq, seq_len, ref, ref_len, threads=1):
    """Local alignment counts as xb_align_counts computes them (the contract at the top of c/align_exact.c):
    seq (N, Ts) / ref (N, Tr) int8 rows with lengths (N,) -> (N, 5) int32 (score, eq, x, ins, del).
    threads > 1 spreads the pairs over host threads (ctypes releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    s, r = np.ascontiguousarray(seq, dtype=np.int8), np.ascontiguousarray(ref, dtype=np.int8)
    sl, rl = np.ascontiguousarray(seq_len, dtype=np.int32), np.ascontiguousarray(ref_len, dtype=np.int32)
    N = len(sl)
    out = np.zeros((N, 5), dtype=np.int32)
    threads = max(1, min(threads, N))
    bounds = [(N * i // threads, N * (i + 1) // threads) for i in range(threads)]
    fn = lib().xbo_align_counts_range

    def work(b):
        return fn(_p(s), s.shape[1], _p(sl), _p(r), r.shape[1], _p(rl), b[0], b[1], _p(out))

    with ThreadPoolExecutor(threads) as ex:
        rcs = list(ex.map(work, bounds))
    assert all(rc == 0 for rc in rcs), rcs
    return out


def rows(strings, width=None):
    """Left-packed (N, width) int8 rows and (N,) int32 lengths of byte strings (str or bytes)."""
    bs = [x.encode() if isinstance(x, str) else bytes(x) for x in strings]
    width = max([len(b) for b in bs] + [1]) if width is None else width
    out = np.zeros((len(bs), width), dtype=np.int8)
    for i, b in enumerate(bs):
        out[i, :len(b)] = np.frombuffer(b, dtype=np.int8)
    return out, np.array([len(b) for b in bs], dtype=np.int32)


def align_strings(seqs, refs, threads=1):
    """align_counts of string pairs: (N, 5) int32."""
    s, sl = rows(seqs)
    r, rl = rows(refs)
    return align_counts(s, sl, r, rl, threads)
