"""CPU checks of the float64 stage references in oracle/train_stages.py that tests/test_gpu_train_stages.py compares the
encoder backward's stages with: the step-by-step LSTM backward without rounding equals autograd through the plain layer
and through torch's own LSTM op to float64 precision, and fp32 autograd to fp32 precision; the head and stem references
equal fp32 autograd of the oracle modules, and the stem written as the kernels compute it equals the stem's autograd
without rounding.  The CTC-CRF loss reference (what tests/test_gpu_ctc_loss.py compares xb_ctc_crf_loss_fwd / _bwd with)
equals fp32 autograd through the oracle's ctc_loss, central differences and float64 autograd of the restated seqdist
scans, and keeps the kernels' contract for targets no alignment reaches."""
import pytest
import torch

from oracle import bonito_oracle as bo
from oracle import train_stages as ts

F64 = torch.float64


def _layer(seed, T, N, F):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(T, N, F, generator=g, dtype=F64)
    w_ih = torch.randn(4 * F, F, generator=g, dtype=F64) * F ** -0.5
    w_hh = torch.randn(4 * F, F, generator=g, dtype=F64) * 0.5 * F ** -0.5
    b = torch.randn(4 * F, generator=g, dtype=F64) * 0.5
    dy = torch.randn(T, N, F, generator=g, dtype=F64)
    return x, w_ih, w_hh, b, dy


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('T,N,F', [(7, 3, 8), (1, 2, 8), (2, 5, 16)])
def test_lstm_matched_without_rounding_is_autograd(T, N, F, reverse):
    x, w_ih, w_hh, b, dy = _layer(3 + T, T, N, F)
    y, *ref = ts.lstm_backward(x, w_ih, w_hh, b, dy, reverse)
    got = ts.lstm_backward_matched(x, y, w_ih, w_hh, b, dy, reverse, rounded=False)
    for a, r in zip(got, ref):
        assert _rel(a, r) <= 1e-12
    if T == 1:
        assert torch.equal(ref[1], torch.zeros_like(ref[1]))         # no step pair: dW_hh is exactly zero
    # torch's own LSTM op (what the reference executes), in float64
    ps = [t.clone().requires_grad_() for t in (x, w_ih, w_hh, b)]
    y2 = bo.lstm_layer_library(ps[0], ps[1], ps[2], ps[3], torch.zeros_like(ps[3]), reverse)
    assert _rel(y2.detach(), y) <= 1e-12
    y2.backward(dy)
    lib = [ps[1].grad, ps[2].grad, ps[3].grad, ps[0].grad]
    for a, r in zip(got, lib):
        assert _rel(a, r) <= 1e-12
    # bo's fp32 modules through fp32 autograd
    ps = [t.float().requires_grad_() for t in (x, w_ih, w_hh, b)]
    bo.lstm_layer(ps[0], ps[1], ps[2], ps[3], torch.zeros_like(ps[3]), reverse).backward(dy.float())
    for a, r in zip(got, [ps[1].grad, ps[2].grad, ps[3].grad, ps[0].grad]):
        assert _rel(a, r.double()) <= 1e-5


def test_lstm_rounding_is_small_and_direction_matters():
    x, w_ih, w_hh, b, dy = _layer(11, 6, 4, 16)
    dy = dy.bfloat16().double()
    y, *ref = ts.lstm_backward(x, w_ih, w_hh, b, dy, True)
    y = y.half().double()
    rounded = ts.lstm_backward_matched(x, y, w_ih, w_hh, b, dy, True)
    for a, r in zip(rounded, ref):
        assert 0 < _rel(a, r) <= 2e-2
    assert torch.equal(rounded[3], rounded[3].bfloat16().double())       # the outgoing gradient is bf16
    other = ts.lstm_backward_matched(x, y, w_ih, w_hh, b, dy, False)
    assert _rel(other[1], rounded[1]) > 0.1


def test_head_and_stem_references_match_fp32_autograd():
    sd = bo.reference_state_dict(n_base=4, seed=5, features=32)
    g = torch.Generator().manual_seed(2)
    T, N, n_base = 6, 3, 4
    x = torch.randn(T, N, 32, generator=g)
    w, b = sd['encoder.9.linear.weight'], sd['encoder.9.linear.bias']
    ds = torch.randn(T, N, 4 ** 3 * 5, generator=g)
    dw, db, dx = ts.crf_head_backward(x, w, b, ds, n_base)
    ps = [t.clone().requires_grad_() for t in (w, b, x)]
    bo.crf_head({'encoder.9.linear.weight': ps[0], 'encoder.9.linear.bias': ps[1]}, ps[2], n_base).backward(ds)
    for a, r in zip((dw, db, dx), ps):
        assert _rel(a, r.grad.double()) <= 1e-5
    # blank columns carry a constant: a cotangent only there has no gradient at all
    blank = torch.zeros_like(ds).reshape(T, N, -1, n_base + 1)
    blank[..., 0] = 1.0
    assert all(not t.any() for t in ts.crf_head_backward(x, w, b, blank.reshape(T, N, -1), n_base))
    sig = torch.randn(N, 50, generator=g)
    conv = [sd['encoder.%d.conv.%s' % (i, k)] for i in range(3) for k in ('weight', 'bias')]
    dy = torch.randn(10, N, 32, generator=g)
    got = ts.conv_stem_backward(sig, *conv, dy)
    ps = [t.clone().requires_grad_() for t in conv]
    keys = ['encoder.%d.conv.%s' % (i, k) for i in range(3) for k in ('weight', 'bias')]
    bo.conv_stem(dict(zip(keys, ps)), sig[:, None]).permute(2, 0, 1).backward(dy)
    for a, r in zip(got, ps):
        assert a.shape == r.shape and _rel(a, r.grad.double()) <= 1e-5
    # the stem written as the kernels compute it (im2col GEMM for conv3): without rounding, the exact backward
    exact = ts.conv_stem_backward_matched(sig, *conv, dy, rounded=False)
    for a, r in zip(exact, got):
        assert a.shape == r.shape and _rel(a, r) <= 1e-12
    rounded = ts.conv_stem_backward_matched(sig, *conv, dy)
    for a, r in zip(rounded, got):
        assert 0 < _rel(a, r) <= 2e-2


def test_held_weights():
    w = torch.tensor([1.0 + 2 ** -12, 3.0e-3, -7.77])
    assert torch.equal(ts.held(w), w.half().double())
    assert torch.equal(ts.held(w, bf16=True), w.bfloat16().double())
    assert torch.equal(ts.held_bwd(w), w.bfloat16().double())


# ----------------------------------------------------------------------------------------------------------- CTC-CRF loss
def _ctc_case(n_base, T=40, N=4, lo=8, hi=20, seed=0):
    from make_golden import synthetic_scores, synthetic_targets
    s = synthetic_scores(7 + n_base + seed, T, N, n_base)
    tg, tl = synthetic_targets(3 + n_base + seed, N, n_base, lo, hi)
    w = torch.tensor([1.0, 0.0, -0.5, 0.25, 0.7, -2.0][:N])
    return s, tg, tl, w


def _ctc_loss_f64(crf, s, tg, tl, normalise):
    """CTC_CRF.ctc_loss(reduction='none') restated in float64 (bo.CRF.ctc_loss casts to float32), for autograd."""
    if normalise:
        s = crf.normalise(s)
    stay, move = crf.prepare_ctc_scores(s, tg, dtype=F64)
    return -crf.simple_logZ(stay, move, tl + 1 - crf.state_len) / tl


@pytest.mark.parametrize('normalise', [True, False])
@pytest.mark.parametrize('n_base', [4, 5, 6])
def test_ctc_reference_is_fp32_autograd(n_base, normalise):
    """The float64 loss and gradient equal autograd through the fp32 oracle (bo.CRF.ctc_loss) within fp32 rounding."""
    from make_golden import ALPHABETS
    s, tg, tl, w = _ctc_case(n_base)
    loss, d = ts.ctc_loss_backward(s, tg, tl, w, n_base, normalise=normalise)
    assert loss.dtype == F64 and d.dtype == F64 and d.shape == s.shape
    sr = s.clone().requires_grad_()
    ref = bo.CRF(3, ALPHABETS[n_base]).ctc_loss(sr, tg, tl, reduction='none', normalise_scores=normalise)
    (ref * w).sum().backward()
    assert ((loss - ref.double()).abs() / loss.abs()).max().item() <= 2e-6
    assert _rel(d, sr.grad.double()) <= 5e-5
    assert (d - sr.grad.double()).abs().max().item() <= 5e-6
    assert not d[:, 1].any()                                  # grad_loss 0: no gradient at all


@pytest.mark.parametrize('normalise', [True, False])
def test_ctc_reference_finite_differences(normalise):
    """In float64 the gradient is the derivative of the loss: central differences on elements of the target's stay and
    move edges, of edges off the target, and of the blank column."""
    n_base = 5
    s, tg, tl, w = _ctc_case(n_base, T=12, N=2, lo=5, hi=9, seed=4)
    s = s.double()
    _, d = ts.ctc_loss_backward(s, tg, tl, w, n_base, normalise=normalise)
    t0 = tg[0].clamp_min(1) - 1
    stay0 = int(((t0[0] * n_base + t0[1]) * n_base + t0[2]) * (n_base + 1))
    move1 = int(((t0[1] * n_base + t0[2]) * n_base + t0[3]) * (n_base + 1) + t0[0] + 1)
    eps = 1e-6
    for t, n, e in [(0, 0, stay0), (1, 0, move1), (5, 0, move1), (11, 0, stay0), (3, 0, 17), (7, 0, 6 * 40), (2, 1, 1)]:
        sp, sm = s.clone(), s.clone()
        sp[t, n, e] += eps
        sm[t, n, e] -= eps
        lp = (ts.ctc_loss_backward(sp, tg, tl, w, n_base, normalise=normalise)[0] * w.double()).sum()
        lm = (ts.ctc_loss_backward(sm, tg, tl, w, n_base, normalise=normalise)[0] * w.double()).sum()
        fd = ((lp - lm) / (2 * eps)).item()
        assert abs(fd - d[t, n, e].item()) <= 1e-7 * max(1.0, abs(fd)), (t, n, e, fd, d[t, n, e].item())


@pytest.mark.parametrize('n_base', [4, 5, 6])
def test_ctc_reference_closed_form_and_zero_sum(n_base):
    """The gradient is (P_den - P_num) * grad_loss / length, with P_den = d sum(logZ) / d scores and P_num the gradient of
    the alignment lattice's log-sum, both by float64 autograd through the restated seqdist scans; it equals float64
    autograd of the whole loss; and with normalise it sums to zero over the edges of every step, since both posteriors
    sum to one there."""
    from make_golden import ALPHABETS
    s, tg, tl, w = _ctc_case(n_base, T=30, N=3, lo=6, hi=15, seed=9)
    s = s.double()
    crf = bo.CRF(3, ALPHABETS[n_base])
    loss, d = ts.ctc_loss_backward(s, tg, tl, w, n_base)
    sr = s.clone().requires_grad_()
    ref = _ctc_loss_f64(crf, sr, tg, tl, True)
    assert _rel(loss, ref.detach()) <= 1e-14
    (ref * w.double()).sum().backward()
    assert _rel(d, sr.grad) <= 1e-12
    sr = s.clone().requires_grad_()
    p_den = torch.autograd.grad(crf.logZ(sr).sum(), sr)[0]
    assert _rel(p_den, crf.posteriors(s)) <= 1e-12
    sr = s.clone().requires_grad_()
    stay, move = crf.prepare_ctc_scores(sr, tg, dtype=F64)
    p_num = torch.autograd.grad(crf.simple_logZ(stay, move, tl - 2).sum(), sr)[0]
    assert _rel(d, (p_den - p_num) * (w.double() / tl)[:, None]) <= 1e-12
    assert d.sum(2).abs().max().item() <= 1e-13
    assert p_num.sum(2).sub(1).abs().max().item() <= 1e-12
    _, d_raw = ts.ctc_loss_backward(s, tg, tl, w, n_base, normalise=False)
    assert _rel(d_raw, -p_num * (w.double() / tl)[:, None]) <= 1e-12


def test_ctc_reference_infeasible_targets():
    """The kernels' contract for targets no alignment reaches: loss = 1e38 / length, and a gradient of P_den only (with
    normalise) or none at all; the other sequences of the batch are unaffected."""
    n_base = 5
    T = 6
    s, tg, tl, w = _ctc_case(n_base, T=T, N=5, lo=4, hi=T + 4, seed=2)
    tl = torch.tensor([T + 4, 2, 1, 5, T + 3])                # too many moves, len < state_len (x2), feasible (x2)
    w = torch.tensor([0.5, 1.0, -1.0, 0.25, 2.0])
    crf = bo.CRF(3, ['N', 'A', 'C', 'G', 'T', 'X'])
    for normalise in (True, False):
        loss, d = ts.ctc_loss_backward(s, tg, tl, w, n_base, normalise=normalise)
        assert torch.allclose(loss[:3], 1e38 / tl[:3].double(), rtol=1e-15, atol=0)
        assert torch.isfinite(d).all()
        p_den = crf.posteriors(s.double()) if normalise else torch.zeros_like(d)
        assert torch.equal(d[:, :3], p_den[:, :3] * (w[:3].double() / tl[:3])[:, None])
        alone, d_alone = ts.ctc_loss_backward(s[:, 3:], tg[3:], tl[3:], w[3:], n_base, normalise=normalise)
        assert torch.equal(loss[3:], alone) and torch.equal(d[:, 3:], d_alone)
    # len = T + 3: a single alignment that moves at every step; its loss is the sum of those move scores
    t0 = tg[4].clamp_min(1) - 1
    st = [int((t0[j] * n_base + t0[j + 1]) * n_base + t0[j + 2]) for j in range(T + 1)]
    path = sum(s[t, 4, st[t + 1] * (n_base + 1) + int(t0[t]) + 1].double() for t in range(T))
    loss, _ = ts.ctc_loss_backward(s, tg, tl, w, n_base, normalise=False)
    assert abs(loss[4].item() + path.item() / (T + 3)) <= 1e-14
