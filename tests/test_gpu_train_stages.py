"""The encoder backward one stage at a time (xb_encoder_bwd_stages: 6 CRF head, 5 .. 1 LSTM layers 4 .. 0, 0 stem), each
stage against a float64 reference (oracle/train_stages.py) on the stage's exact 16-bit inputs.

The inputs come from the inference hooks (Handle.conv_stem, Handle.lstm, Handle.crf_head); that their chain gives the
training forward's scores bit for bit is asserted every time, and is the evidence that these are the tensors the training
forward kept.  Cotangents are bf16-representable: drawn in fp32, rounded to bf16 and passed as the bf16 dy_top.

Every gradient tensor is compared by its relative error in the 2-norm and by its cosine to the reference (>= COS_TOL), as
test_gpu_train.py does, but per stage, and the tight bound of each stage is at least 5x tighter than the end-to-end 3e-2:
  * LSTM layer: against the rounding-matched reference (it rounds where the kernels round, so what is left is the
    accumulation order) with MATCHED_TOL, and against the plain float64 autograd reference with PLAIN_TOL;
  * CRF head: against the plain float64 reference with HEAD_TOL;
  * stem: against the rounding-matched reference with STEM_TOL.  Against the plain reference it cannot meet a tight bound:
    the kernels round conv3's im2col rows (the conv2 output) to fp16 and conv3's gradients to bf16, and where a gradient
    is a sum that mostly cancels -- conv1's bias with dy at the last step only -- those roundings move it by ~1 %, while
    the rounding-matched reference, which makes the same roundings, agrees to 7e-4.  The plain comparison keeps the
    end-to-end bound, STEM_PLAIN_TOL.

Largest errors observed on a B200 (1000 W power limit) over every case of this file -- T = 800 and the T = 1, 2 edges,
fp16 and bf16 handles, N = 8 and 136, all layers, n_base 4..6, every stem length and cotangent -- and the bounds, each a
small multiple of them:
  LSTM vs rounding-matched   rel 2.2e-3 (dy_bottom; dW_ih 1.0e-3, dW_hh 8.2e-4, db 8.2e-4)    MATCHED_TOL     5e-3
  LSTM vs plain float64      rel 3.0e-3 (dy_bottom; dW_ih 2.3e-3, dW_hh 2.4e-3, db 1.5e-3)    PLAIN_TOL       6e-3
  head vs plain float64      rel 2.9e-3 (dy_bottom; dW 2.5e-3, db 1.8e-3)                     HEAD_TOL        6e-3
  stem vs rounding-matched   rel 6.8e-4 (conv1 bias, dy at the last step; conv3 weight 1.0e-4) STEM_TOL        2e-3
  stem vs plain float64      rel 1.3e-2 (conv1 bias, dy at the last step; all others <= 5.7e-3) STEM_PLAIN_TOL  3e-2
  smallest cosine            0.99996 (stem vs plain), >= 0.9999976 for every other comparison  COS_TOL    0.9999
"""
import pytest
import torch

from make_golden import ALPHABETS, REF_SCALE, synthetic_signal
from oracle import bonito_oracle as bo
from oracle import train_stages as ts

pytestmark = pytest.mark.gpu

COS_TOL = 0.9999
MATCHED_TOL = 5e-3
PLAIN_TOL = 6e-3
HEAD_TOL = 6e-3
STEM_TOL = 2e-3
STEM_PLAIN_TOL = 3e-2
LSTM_KEYS = ('weight_ih_l0', 'weight_hh_l0', 'bias_ih_l0')


def _err(got, ref):
    a, b = got.double().flatten(), ref.double().flatten().to(got.device)
    rel = ((a - b).norm() / b.norm().clamp_min(1e-30)).item()
    cos = (torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)).item()
    return rel, cos


def _check(what, got, ref, tol):
    rel, cos = _err(got, ref)
    print('%-44s rel %.2e  cos %.7f  (bound %.0e)' % (what, rel, cos, tol))
    assert rel <= tol and cos >= COS_TOL, (what, rel, cos)


def _bf16_cot(seed, *shape, device='cuda'):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g).bfloat16().to(device)


_CACHE = {}


def _setup(n_base, N, T, bf16=False):
    """Handle after one training forward on synthetic signal, with the inputs of every stage from the inference hooks:
    (h, sd, signal, xs) where xs[0] is the stem output and xs[l + 1] the output of LSTM layer l.  Keeps the last one."""
    key = (n_base, N, T, bf16)
    if key not in _CACHE:
        for v in _CACHE.values():
            v[0].close()
        _CACHE.clear()
        torch.cuda.empty_cache()
        from xna_basecaller_b200._lib import Handle
        sd = bo.reference_state_dict(n_base=n_base, seed=12, **REF_SCALE)
        x = synthetic_signal(41 + T + N, N, 5 * T).cuda()
        h = Handle(ALPHABETS[n_base], 3, max_N=N, max_T=T, train=True, bf16=bf16)
        h.load_weights(sd)
        xs = [h.conv_stem(x)]
        for l in range(5):
            xs.append(h.lstm(l, xs[-1], bo.LSTM_DIRECTIONS[l]))
        scores = h.encoder_train(x)
        assert torch.equal(h.crf_head(xs[5]), scores)
        _CACHE[key] = (h, sd, x, xs)
    return _CACHE[key]


def _lstm_refs(sd, xs, l, dy, bf16):
    p = 'encoder.%d.rnn.' % (l + 4)
    w_ih, w_hh = ts.held(sd[p + 'weight_ih_l0'], bf16).cuda(), ts.held(sd[p + 'weight_hh_l0'], bf16).cuda()
    b = (sd[p + 'bias_ih_l0'] + sd[p + 'bias_hh_l0']).double().cuda()
    rev = bo.LSTM_DIRECTIONS[l]
    matched = ts.lstm_backward_matched(xs[l], xs[l + 1], w_ih, w_hh, b, dy, rev,
                                       w_ih_t=ts.held_bwd(sd[p + 'weight_ih_l0']).cuda(),
                                       w_hh_t=ts.held_bwd(sd[p + 'weight_hh_l0']).cuda())
    return matched, lambda: ts.lstm_backward(xs[l], w_ih, w_hh, b, dy, rev)[1:]


def _lstm_stage(h, l, dy):
    g, dyb = h.encoder_backward_stages(l + 1, l + 1, dy_top=dy)
    p = 'encoder.%d.rnn.' % (l + 4)
    assert sorted(g) == sorted(p + k for k in LSTM_KEYS + ('bias_hh_l0',))
    assert torch.equal(g[p + 'bias_hh_l0'], g[p + 'bias_ih_l0'])
    return [g[p + k] for k in LSTM_KEYS] + [dyb]


# ----------------------------------------------------------------------------------------------------------- LSTM
# N = 136: two row tiles of the BPTT step kernel, the second clipped at the batch edge
@pytest.mark.parametrize('bf16', [False, True])
@pytest.mark.parametrize('N,T', [(8, 800), (136, 800), (8, 2)])
def test_lstm_stage_matches_float64(N, T, bf16):
    h, sd, _, xs = _setup(5, N, T, bf16)
    names = ('dW_ih', 'dW_hh', 'db', 'dy_bottom')
    for l in range(5):
        dy = _bf16_cot(100 + l, T, N, 768)
        got = _lstm_stage(h, l, dy)
        matched, plain = _lstm_refs(sd, xs, l, dy, bf16)
        for name, a, r in zip(names, got, matched):
            _check('layer %d %s vs rounding-matched' % (l, name), a, r, MATCHED_TOL)
        for name, a, r in zip(names, got, plain()):
            _check('layer %d %s vs plain float64' % (l, name), a, r, PLAIN_TOL)


def test_lstm_stage_structural_zeros():
    """Exact zeros that hold at any precision: chunks do not mix, a step's gradient does not reach the steps the forward
    ran after it."""
    N, T = 136, 200
    h, _, _, _ = _setup(5, N, T)
    for l in (0, 1):
        for c in (3, 130):                       # one chunk of each BPTT row tile
            dy = torch.zeros(T, N, 768, dtype=torch.bfloat16, device='cuda')
            dy[:, c] = _bf16_cot(7 + c, T, 768)
            _, _, _, dyb = _lstm_stage(h, l, dy)
            others = torch.ones(N, dtype=torch.bool)
            others[c] = False
            assert not dyb[:, others.cuda()].any() and dyb[:, c].any()
        t0 = 77
        dy = torch.zeros(T, N, 768, dtype=torch.bfloat16, device='cuda')
        dy[t0] = _bf16_cot(5, N, 768)
        _, _, _, dyb = _lstm_stage(h, l, dy)
        after = slice(0, t0) if bo.LSTM_DIRECTIONS[l] else slice(t0 + 1, T)
        assert not dyb[after].any() and dyb[t0].any()


@pytest.mark.parametrize('bf16', [False, True])
def test_lstm_stage_single_step(bf16):
    """T = 1 (L = 5): no step has a predecessor, so dW_hh is exactly zero."""
    h, sd, _, xs = _setup(5, 8, 1, bf16)
    for l in range(5):
        dy = _bf16_cot(30 + l, 1, 8, 768)
        got = _lstm_stage(h, l, dy)
        assert not got[1].any()
        matched, _ = _lstm_refs(sd, xs, l, dy, bf16)
        for name, a, r in zip(('dW_ih', 'db', 'dy_bottom'), (got[0], got[2], got[3]), (matched[0], matched[2], matched[3])):
            _check('T=1 layer %d %s' % (l, name), a, r, MATCHED_TOL)


@pytest.mark.parametrize('l', [0, 1])
def test_lstm_stage_time_edges(l):
    """dy_top non-zero only at the forward's first, then only at its last step, T = 800: a step lost or shifted at either
    end of the BPTT walk or of dW_hh's time-shifted contraction changes these gradients by 100 %, not by 1/T."""
    N, T = 8, 800
    h, sd, _, xs = _setup(5, N, T)
    first, last = (T - 1, 0) if bo.LSTM_DIRECTIONS[l] else (0, T - 1)
    for what, t in (('first', first), ('last', last)):
        dy = torch.zeros(T, N, 768, dtype=torch.bfloat16, device='cuda')
        dy[t] = _bf16_cot(50 + t, N, 768)
        got = _lstm_stage(h, l, dy)
        matched, _ = _lstm_refs(sd, xs, l, dy, False)
        if what == 'first':
            assert not got[1].any()              # dz is non-zero at the first step only, which has no h_prev
        else:
            _check('layer %d dW_hh, dy at the last step' % l, got[1], matched[1], MATCHED_TOL)
        _check('layer %d dW_ih, dy at the %s step' % (l, what), got[0], matched[0], MATCHED_TOL)
        _check('layer %d dy_bottom, dy at the %s step' % (l, what), got[3], matched[3], MATCHED_TOL)


# ----------------------------------------------------------------------------------------------------------- head
@pytest.mark.parametrize('n_base,N', [(4, 8), (5, 8), (6, 8), (4, 136), (5, 136), (6, 136)])
def test_head_stage_matches_float64(n_base, N):
    T = 800
    h, sd, _, xs = _setup(n_base, N, T)
    C, NZ = n_base ** 3, n_base + 1
    ds = torch.randn(T, N, C * NZ, generator=torch.Generator().manual_seed(n_base)).cuda() * 1e-2
    g, dyb = h.encoder_backward_stages(6, 6, dscores=ds)
    assert sorted(g) == ['encoder.9.linear.bias', 'encoder.9.linear.weight']
    ref = ts.crf_head_backward(xs[5], ts.held(sd['encoder.9.linear.weight']).cuda(), sd['encoder.9.linear.bias'].cuda(),
                               ds, n_base)
    for name, a, r in zip(('dW', 'db', 'dy_bottom'), (g['encoder.9.linear.weight'], g['encoder.9.linear.bias'], dyb), ref):
        _check('head n_base %d N %d %s' % (n_base, N, name), a, r, HEAD_TOL)
    # the blank scores are constants: a gradient only there reaches nothing
    blank = torch.zeros(T, N, C, NZ, device='cuda')
    blank[..., 0] = 1.0
    g, dyb = h.encoder_backward_stages(6, 6, dscores=blank.reshape(T, N, -1))
    assert not dyb.any() and not any(v.any() for v in g.values())


# ----------------------------------------------------------------------------------------------------------- stem
@pytest.fixture(scope='module')
def stem_handle():
    from xna_basecaller_b200._lib import Handle
    sd = bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE)
    h = Handle(ALPHABETS[5], 3, max_N=8, max_T=800, train=True)
    h.load_weights(sd)
    yield h, sd
    h.close()


# L around and across conv2_bwd_kernel's 256-position tiles; 5 is one step
@pytest.mark.parametrize('L', [5, 250, 260, 515, 4000])
@pytest.mark.parametrize('int16', [False, True])
def test_stem_stage_matches_float64(stem_handle, L, int16):
    h, sd = stem_handle
    N, T = 8, L // 5
    x = synthetic_signal(L, N, L)[:, 0]
    if int16:
        x = torch.round(x * 50).to(torch.int16)      # integers: exactly the same values as fp32
    h.encoder_train(x.cuda())
    conv = [sd['encoder.%d.conv.%s' % (i, k)].cuda() for i in range(3) for k in ('weight', 'bias')]
    conv[4] = ts.held(sd['encoder.2.conv.weight']).cuda()
    keys = ['encoder.%d.conv.%s' % (i, k) for i in range(3) for k in ('weight', 'bias')]
    dense = _bf16_cot(L, T, N, 768)
    for where in ('all', 'first', 'last'):           # the first and last steps: conv3's window reaches the zero padding
        dy = dense
        if where != 'all':
            dy = torch.zeros_like(dense)
            t = 0 if where == 'first' else T - 1
            dy[t] = dense[t]
        g, dyb = h.encoder_backward_stages(0, 0, dy_top=dy)
        assert dyb is None and sorted(g) == sorted(keys)
        what = 'stem L %d %s dy %s ' % (L, 'int16' if int16 else 'fp32', where)
        matched = ts.conv_stem_backward_matched(x.cuda(), *conv, dy, w3_t=ts.held_bwd(sd['encoder.2.conv.weight']).cuda())
        for k, r in zip(keys, matched):
            _check(what + k + ' vs rounding-matched', g[k], r, STEM_TOL)
        for k, r in zip(keys, ts.conv_stem_backward(x.cuda(), *conv, dy)):
            _check(what + k + ' vs plain float64', g[k], r, STEM_PLAIN_TOL)


# ----------------------------------------------------------------------------------------------------------- whole backward
def _same_grads(a, b):
    """LSTM weight gradients come from plain tile GEMMs: equal bit for bit.  The others end in fp32 atomic adds (column sums,
    split-K partials, per-block weight sums) whose order varies from run to run: equal to that reordering's size."""
    assert sorted(a) == sorted(b)
    for k in a:
        if k.endswith(('weight_ih_l0', 'weight_hh_l0')):
            assert torch.equal(a[k], b[k]), k
        else:
            assert ((a[k] - b[k]).double().norm() / b[k].double().norm().clamp_min(1e-30)).item() <= 1e-5, k


@pytest.mark.parametrize('bf16', [False, True])
def test_stages_compose_to_the_whole_backward(bf16):
    from xna_basecaller_b200._lib import Handle
    n_base, N, L = 5, 16, 800
    sd = bo.reference_state_dict(n_base=n_base, seed=12, **REF_SCALE)
    h = Handle(ALPHABETS[n_base], 3, max_N=N, max_T=L // 5, train=True, bf16=bf16)
    h.load_weights(sd)
    x = synthetic_signal(77, N, L)
    scores = h.encoder_train(x.cuda())
    ds = torch.randn(scores.shape, generator=torch.Generator().manual_seed(4)).cuda() * 1e-2
    whole = h.encoder_backward(ds)
    chained, dy = h.encoder_backward_stages(6, 6, dscores=ds)
    for k in range(5, -1, -1):
        g, dy = h.encoder_backward_stages(k, k, dy_top=dy)
        assert not set(g) & set(chained)
        chained.update(g)
    _same_grads(chained, whole)
    # two ranges that split the walk between LSTM layers
    upper, dy = h.encoder_backward_stages(6, 3, dscores=ds)
    lower, _ = h.encoder_backward_stages(2, 0, dy_top=dy)
    _same_grads(dict(upper, **lower), whole)
    # the backward keeps the saved state: a second call gives the same gradients
    _same_grads(h.encoder_backward(ds), whole)
    # int16 signal: the gradients of the same values as fp32
    x16 = torch.round(x * 50).to(torch.int16)
    s16 = h.encoder_train(x16.cuda())
    g16 = h.encoder_backward(ds)
    assert torch.equal(h.encoder_train(x16.float().cuda()), s16)
    _same_grads(g16, h.encoder_backward(ds))
    h.close()


def test_stage_ranges_are_checked():
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=8, max_T=20, train=True)
    h.load_weights(bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE))
    x = synthetic_signal(3, 8, 100).cuda()
    h.encoder_train(x)
    dy = torch.zeros(20, 8, 768, dtype=torch.bfloat16, device='cuda')
    for top, bottom in ((7, 0), (2, 3), (0, -1)):
        with pytest.raises(RuntimeError, match=r'\(-1\)'):
            h.encoder_backward_stages(top, bottom, dy_top=dy)
    with pytest.raises(RuntimeError, match=r'\(-1\)'):
        h.encoder_backward_stages(3, 3)                           # no dy_top
    with pytest.raises(RuntimeError, match=r'\(-1\)'):
        h.encoder_backward_stages(6, 5)                           # no dscores
    h.encoder_train(x, dropout_p=[0.1] * 7, seed=5)
    with pytest.raises(RuntimeError, match=r'\(-4\)'):
        h.encoder_backward_stages(3, 3, dy_top=dy)
    h.close()


def test_backward_times_the_head_and_stem_kernels():
    """xb_stage_times row train_head_conv_bwd: the CRF head's and the convolution stem's own kernels, timed in every
    backward (the transpositions and GEMMs around them have rows of their own)."""
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=8, max_T=20, train=True)
    h.load_weights(bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE))
    scores = h.encoder_train(synthetic_signal(3, 8, 100).cuda())
    ds = torch.randn(scores.shape, generator=torch.Generator().manual_seed(6)).cuda() * 1e-2
    h.set_profiling(True)
    h.stage_times()
    h.encoder_backward(ds)
    ms, spans = h.stage_times()['train_head_conv_bwd']
    h.set_profiling(False)
    h.close()
    assert spans > 0 and ms > 0
