"""CPU restatement of the reference's per-read signal pre-processing (SURVEY section 8f, N2).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): checker for the CUDA kernel in csrc/preprocess.cu.

Follows ub-bonito/bonito/fast5.py: Read.__init__ :88-100 (DAC -> pA scaling, trim, med/MAD normalisation, short reads by
the noisiest section), trim :149-172, and bonito/util.py med_mad / norm_by_noisiest_section (the helpers fast5.py
imports).  Pinned against those very functions through tests/golden/preprocess.npz (tests/test_cpu_preprocess.py).

Arithmetic: float32 throughout, as numpy >= 2 evaluates the reference's expressions (a float32 scalar times a Python
float stays float32).  The reference's pinned numpy 1.19.5 promoted `median * 1.4826` and the trim threshold to float64
before rounding back to float32 for the array operations; the two differ by at most one ulp of mad / threshold.  The
scipy find_peaks(noise, width=...) step of norm_by_noisiest_section acts on a 0/1 array whose ends are forced to 0, where
it reduces to: every maximal run of ones is a peak, its width is the run length, left_base / right_base are the zeros
next to the run -- restated here as run lengths (checked against scipy in the test).
"""
import numpy as np

F = np.float32
MAD_FACTOR = F(1.4826)
EPS = np.finfo(np.float32).eps
TRIM_WINDOW, TRIM_FACTOR, TRIM_MIN_ELEMENTS, MIN_TRIM = 40, F(2.4), 3, 10
HEAD = 8000                      # samples inspected by trim; reads no longer than this use the noisiest section
NOISE_WINDOW, NOISE_DIV = 100, F(6.0)


def scale(raw, scaling, offset):
    """fast5.py:88-89: float32(scaling * (raw + offset)), the product in float64."""
    return (np.float64(scaling) * (raw.astype(np.int64) + int(offset))).astype(np.float32)


def med_mad(x):
    med = np.median(x)
    mad = F(F(np.median(np.abs(x - med))) * MAD_FACTOR) + F(EPS)
    return F(med), F(mad)


def trim(head):
    """fast5.py:149-172 on scaled[:8000]; returns the trim start."""
    signal = head[MIN_TRIM:]
    if len(signal) == 0:
        return MIN_TRIM
    med, mad = med_mad(signal[-(TRIM_WINDOW * 100):])
    threshold = F(med + F(mad * TRIM_FACTOR))
    seen_peak = False
    for pos in range(len(signal) // TRIM_WINDOW):
        window = signal[pos * TRIM_WINDOW:(pos + 1) * TRIM_WINDOW]
        if np.count_nonzero(window > threshold) > TRIM_MIN_ELEMENTS or seen_peak:
            seen_peak = True
            if window[-1] > threshold:
                continue
            return min((pos + 1) * TRIM_WINDOW + MIN_TRIM, len(signal))
    return MIN_TRIM


def noisiest_region(signal):
    """[a, b) of the samples norm_by_noisiest_section takes its med/MAD from."""
    n = len(signal)
    threshold = F(signal.std() / NOISE_DIV)
    noise = np.ones(n, dtype=np.int8)
    for w in range(n // NOISE_WINDOW):
        noise[w * NOISE_WINDOW:(w + 1) * NOISE_WINDOW] = 1 if signal[w * NOISE_WINDOW:(w + 1) * NOISE_WINDOW].std() > threshold else 0
    noise[0] = 0
    noise[-1] = 0
    best, best_len, i = None, 0, 0
    while i < n:
        if noise[i]:
            j = i
            while j < n and noise[j]:
                j += 1
            if j - i > best_len:                 # first of the longest runs (np.argmax)
                best, best_len = (i - 1, j), j - i
            i = j
        else:
            i += 1
    return best if best is not None else (0, n)


def preprocess(raw, scaling, offset):
    """One read: int16 DAC values -> (normalised float32 signal, trim_start, med, mad, mode); mode 0 = med/MAD of the whole
    read, 1 = of the noisiest section (<= 8000 samples after trimming), 2 = nothing left."""
    scaled = scale(np.asarray(raw), scaling, offset)
    start = trim(scaled[:HEAD])
    scaled = scaled[start:]
    if len(scaled) == 0:
        return scaled, start, F(0), F(0), 2
    if len(scaled) > HEAD:
        med, mad = med_mad(scaled)
        mode = 0
    else:
        a, b = noisiest_region(scaled)
        med, mad = med_mad(scaled[a:b])
        mode = 1
    return ((scaled - med) / mad).astype(np.float32), start, med, mad, mode
