"""CPU checks of the float64 stage references in oracle/train_stages.py that tests/test_gpu_train_stages.py compares the
encoder backward's stages with: the step-by-step LSTM backward without rounding equals autograd through the plain layer
and through torch's own LSTM op to float64 precision, and fp32 autograd to fp32 precision; the head and stem references
equal fp32 autograd of the oracle modules, and the stem written as the kernels compute it equals the stem's autograd
without rounding."""
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
