"""Signal pre-processing oracle (oracle/preprocess.py) against the reference's own functions: golden outputs generated from
ub-bonito/bonito/fast5.py (tests/golden/preprocess.npz).  Bit-exact: same float32 bits, same trim index."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), 'golden'))
from make_golden import RAW_LENGTHS, RAW_SCALING, synthetic_raw_read

from oracle import preprocess as pp

GOLD = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'preprocess.npz'))


def test_oracle_matches_reference_golden():
    modes = set()
    for i, n in enumerate(RAW_LENGTHS):
        raw = synthetic_raw_read(1000 + i, n, stall=i % 3 != 2)
        signal, start, med, mad, mode = pp.preprocess(raw, RAW_SCALING, -240 + i)
        assert start == int(GOLD['r%d_trim' % i])
        want = GOLD['r%d_signal' % i]
        assert signal.dtype == np.float32 and signal.shape == want.shape
        assert np.array_equal(signal.view(np.uint32), want.view(np.uint32))
        modes.add(mode)
    assert modes == {0, 1}


def test_edge_cases():
    z = np.zeros(0, dtype=np.int16)
    assert pp.preprocess(z, RAW_SCALING, 0)[4] == 2 and len(pp.preprocess(z, RAW_SCALING, 0)[0]) == 0
    assert pp.preprocess(np.arange(7, dtype=np.int16), RAW_SCALING, 3)[4] == 2          # shorter than the minimum trim
    s, start, _, _, mode = pp.preprocess(np.arange(11, dtype=np.int16), RAW_SCALING, 3)  # one sample left
    assert start == 10 and mode == 1 and len(s) == 1
    flat = np.full(9000, 321, dtype=np.int16)                                            # MAD = eps
    s, start, med, mad, mode = pp.preprocess(flat, RAW_SCALING, 0)
    assert mode == 0 and mad == np.finfo(np.float32).eps and np.all(s == 0)

