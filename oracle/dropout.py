"""numpy restatement of the dropout mask contract of the training step (xna_basecaller_b200/csrc/xb_dropout.cuh), and
the fp32 encoder forward with those masks applied where rnn_encoder(drop_rate_bottom=...) puts its Dropout modules
(bonito/crf/model.py rnn_encoder: after each convolution and after LSTM layers 0-3).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Written from the contract, not from the kernels: Philox4x32-10 as
Random123 defines it (known-answer vectors in tests/test_cpu_dropout.py), vectorised over counters with 64-bit products.

PARITY: the masks follow torch.nn.Dropout's distribution (keep with probability 1 - p, scale kept values by 1 / (1 - p)),
not torch's random stream -- parity unpinned against torch's generator.
"""
import numpy as np
import torch

from . import bonito_oracle as bo

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
SITES = 7
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10.  ctr: (..., 4) uint32-valued array, key: (2,) -> (..., 4) uint32."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] for i in range(4)]
    k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(W0)) & MASK32, (k1 + np.uint64(W1)) & MASK32
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1).astype(np.uint32)


def threshold(p):
    """(thr, scale) of probability p, as the library computes them from the float it receives."""
    pf = float(np.float32(p))
    if not 0.0 <= pf < 1.0:
        raise ValueError('dropout probability must lie in [0, 1), got %r' % (p,))
    thr = min(int(np.floor(pf * 2.0 ** 32)), 2 ** 32 - 1)
    return thr, np.float32(1.0 / (1.0 - pf))


def keep(seed, site, p, n):
    """Keep flags (n,) bool of elements 0 .. n-1 of dropout site `site`."""
    thr, _ = threshold(p)
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.stack([q & MASK32, q >> np.uint64(32), np.full_like(q, site), np.zeros_like(q)], axis=-1)
    words = philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)).reshape(-1)[:n]
    return words >= np.uint32(thr) if thr else np.ones(n, dtype=bool)


def mask(seed, site, p, shape):
    """Multiplier tensor (fp32, `shape`, row-major flat index = element index): scale where kept, 0 where dropped."""
    n = int(np.prod(shape))
    _, scale = threshold(p)
    return torch.from_numpy(np.where(keep(seed, site, p, n), scale, np.float32(0)).astype(np.float32).reshape(shape))


def _drop(y, seed, site, p):
    if not p:
        return y
    return y * mask(seed, site, p, tuple(y.shape))


def encoder_forward_dropout(sd, x, n_base, p, seed, scale=5.0, blank_score=2.0):
    """bo.encoder_forward with the masks of the seven sites applied: p = seven probabilities (conv1, conv2, conv3 outputs,
    outputs of LSTM layers 0-3).  Site tensors are indexed as the contract says: (N, C, L) for the first two, (T, N, 768)
    for the rest.  Differentiable (the masks are constants)."""
    y = bo.swish(torch.nn.functional.conv1d(x, sd['encoder.0.conv.weight'], sd['encoder.0.conv.bias'], padding=2))
    y = _drop(y, seed, 0, p[0])
    y = bo.swish(torch.nn.functional.conv1d(y, sd['encoder.1.conv.weight'], sd['encoder.1.conv.bias'], padding=2))
    y = _drop(y, seed, 1, p[1])
    w = sd['encoder.2.conv.weight']
    y = bo.swish(torch.nn.functional.conv1d(y, w, sd['encoder.2.conv.bias'], stride=5, padding=w.shape[-1] // 2))
    y = y.permute(2, 0, 1).contiguous()
    y = _drop(y, seed, 2, p[2])
    for i, (layer, rev) in enumerate(zip(range(4, 9), bo.LSTM_DIRECTIONS)):
        pre = 'encoder.%d.rnn.' % layer
        y = bo.lstm_layer(y, sd[pre + 'weight_ih_l0'], sd[pre + 'weight_hh_l0'], sd[pre + 'bias_ih_l0'],
                          sd[pre + 'bias_hh_l0'], rev)
        if i < 4:
            y = _drop(y, seed, 3 + i, p[3 + i])
    return bo.crf_head(sd, y, n_base, scale, blank_score)
