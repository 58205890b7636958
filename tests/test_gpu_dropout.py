"""GPU tests of dropout in the training step (rnn_encoder(drop_rate_bottom=...); mask contract in csrc/xb_dropout.cuh,
numpy restatement in oracle/dropout.py):

  * the device generator equals the numpy restatement bit for bit;
  * in eval mode a drop_rate_bottom model runs every inference route with the bits of the plain model;
  * with p = 0 on every site the training step is the plain step (same bits, same launches);
  * with p > 0 forward and gradients match an fp32 autograd oracle that applies the numpy masks, at the bounds and shapes
    of test_gpu_train.py::test_encoder_backward_matches_autograd;
  * masks are seeded from torch's CPU generator, one draw per forward, and every backward replays its own forward's masks.
"""
import numpy as np
import pytest
import torch

from make_golden import ALPHABETS, REF_SCALE, synthetic_signal, synthetic_targets
from oracle import bonito_oracle as bo
from oracle import dropout as od
from test_cpu_host import sup_config

pytestmark = pytest.mark.gpu

REL_TOL, COS_TOL = 3e-2, 0.999


def _compare(got, ref):
    worst = {}
    for k, g in ref.items():
        if k.endswith('bias_hh_l0') or g is None:      # frozen at zero in the reference: no gradient of its own
            continue
        a, b = got[k].double().cpu().flatten(), g.double().flatten()
        rel = ((a - b).norm() / b.norm().clamp_min(1e-30)).item()
        cos = (torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)).item()
        worst[k] = (rel, cos)
    return worst


def _model(n_base=5, **encoder):
    from xna_basecaller_b200 import util
    cfg = sup_config(ALPHABETS[n_base])
    cfg['encoder'].update(encoder)
    return util.load_symbol(cfg, 'Model')(cfg)


def _copy_params(src, dst):
    """dst <- src parameter by parameter (the state_dict keys differ: Dropout modules shift the Serial indices)."""
    a, b = list(src.named_parameters()), list(dst.named_parameters())
    assert [n.rsplit('.', 2)[-2:] for n, _ in a] == [n.rsplit('.', 2)[-2:] for n, _ in b]
    with torch.no_grad():
        for (_, p), (_, q) in zip(a, b):
            q.copy_(p)
            q.requires_grad_(p.requires_grad)


def _pair(sd, **drop):
    plain, dropped = _model(), _model(**drop)
    plain.load_state_dict(sd)
    _copy_params(plain, dropped)
    return plain.to('cuda'), dropped.to('cuda')


def _named_grads(model):
    return [(n, p.grad.clone()) for n, p in model.named_parameters() if p.grad is not None]


def _assert_same_grads(ga, gb):
    """Same gradients from the same kernels.  The LSTM weight gradients come from plain tile GEMMs and must be equal bit for
    bit; the bias, convolution and head gradients end in fp32 atomic adds (column sums, split-K partials, per-block weight
    sums), whose order varies from run to run even without dropout, so those are compared at that reordering's size."""
    assert [n.rsplit('.', 2)[-2:] for n, _ in ga] == [n.rsplit('.', 2)[-2:] for n, _ in gb]
    for (n, a), (_, b) in zip(ga, gb):
        if n.endswith(('weight_ih_l0', 'weight_hh_l0')):
            assert torch.equal(a, b), n
        else:
            assert ((a - b).norm() / b.norm().clamp_min(1e-30)).item() <= 1e-5, n


# ---------------------------------------------------------------------------------------------------------- generator
@pytest.mark.parametrize('seed', [0x0123456789abcdef, 0x7ffffffffffffffd])
def test_keep_flags_match_numpy(seed):
    from xna_basecaller_b200 import _lib
    n = 100003                     # not a multiple of the four elements one generator call decides
    for site in range(7):
        for p in (0.1, 0.5, 0.9):
            got = _lib.dropout_keep(seed, site, p, n).cpu().numpy()
            want = od.keep(seed, site, p, n)
            assert np.array_equal(got, want), (site, p, int((got != want).sum()))
            assert abs(got.mean() - (1 - p)) < 0.01


def test_bad_probabilities_are_refused():
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=8, max_T=20, train=True)
    h.load_weights(bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE))
    x = synthetic_signal(3, 8, 100).cuda()
    for p in ([0.1] * 6 + [1.0], [0.1] * 6, [-0.1] + [0.0] * 6):
        with pytest.raises(ValueError):
            h.encoder_train(x, dropout_p=p, seed=1)
    h.close()


# ---------------------------------------------------------------------------------------------------------- eval mode
def test_eval_mode_is_the_plain_model_on_every_route():
    from xna_basecaller_b200 import pipeline
    import importlib
    cb = importlib.import_module('xna_basecaller_b200.crf.basecall')      # the package re-exports basecall()
    from xna_basecaller_b200.training import Trainer
    plain, dropped = _pair(bo.reference_state_dict(n_base=5, seed=11), drop_rate_bottom=0.1)
    plain.eval()
    dropped.eval()
    x = synthetic_signal(21, 8, 1000)
    with torch.no_grad():
        a, b = plain(x.cuda()), dropped(x.cuda())
    assert torch.equal(a, b)
    strings = plain.decode_batch(a)
    assert dropped.decode_batch(b) == strings and any(strings)

    ra, rb = cb.compute_scores(plain, x), cb.compute_scores(dropped, x)
    assert torch.equal(ra['sequence'], rb['sequence']) and torch.equal(ra['qstring'], rb['qstring'])     # host fast path
    pa, pb = cb._collect_scores(*cb._submit_scores(plain, x, 1)), cb._collect_scores(*cb._submit_scores(dropped, x, 1))
    assert torch.equal(pa['sequence'], pb['sequence']) and torch.equal(pa['sequence'], ra['sequence'])  # pipelined

    class Read:
        def __init__(self, rid, sig):
            self.read_id, self.signal = rid, sig

    rs = np.random.RandomState(8)
    sigs = [rs.randn(L).astype(np.float32) for L in (700, 2350, 3100, 999, 4600)]
    reads = lambda: iter([Read(i, s) for i, s in enumerate(sigs)])
    for fn in (lambda m: [r['sequence'] for _, r in cb.basecall(m, reads(), chunksize=1000, overlap=100, batchsize=4)],
               lambda m: [r['sequence'] for _, r in pipeline.basecall_reads(m, reads(), chunksize=1000, overlap=100,
                                                                           batchsize=7, block_reads=3)],
               lambda m: pipeline.ReadSetBasecaller(m, chunksize=1000, overlap=100, batchsize=7).basecall(sigs)[0]):
        sa, sb = fn(plain), fn(dropped)
        assert sa == sb and any(sa)

    tg, tl = synthetic_targets(7, 8, 5, 40, 60)
    va = Trainer(plain, 'cuda').validate_one_step((x, tg, tl))
    vb = Trainer(dropped, 'cuda').validate_one_step((x, tg, tl))
    assert va == vb


# ---------------------------------------------------------------------------------------------------------- p = 0
def test_zero_probabilities_are_the_plain_step():
    plain, dropped = _pair(bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE), drop_rate_bottom=0.1)
    for m in dropped.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    assert sum(isinstance(m, torch.nn.Dropout) for m in dropped.encoder) == 7
    x = synthetic_signal(41, 8, 500).cuda()
    cot = torch.randn(100, 8, 5 ** 3 * 6, generator=torch.Generator().manual_seed(9)).cuda() * 1e-2
    results = []
    for m in (plain, dropped):
        m.train()
        state = torch.get_rng_state()
        counts = []
        for _ in range(2):                 # the second round runs on a warm handle
            m.zero_grad()
            h0 = m.seqdist.engine.handle.launches if m.seqdist.engine.handle else 0
            scores = m(x)
            scores.backward(cot)
            torch.cuda.synchronize()
            counts.append(m.seqdist.engine.handle.launches - h0)
        assert torch.equal(torch.get_rng_state(), state)          # nothing drawn from torch's generator without dropout
        results.append((scores.detach(), _named_grads(m), counts[1]))
    (sa, ga, ca), (sb, gb, cb) = results
    assert torch.equal(sa, sb)
    assert len(ga) == len(gb) == 28 - 5          # bias_hh is frozen
    _assert_same_grads(ga, gb)
    assert ca == cb


# ---------------------------------------------------------------------------------------------------------- parity
@pytest.mark.parametrize('p', [0.1, 0.5])
@pytest.mark.parametrize('n_base,N,L', [(5, 8, 500), (6, 16, 300), (5, 136, 100)])
def test_dropout_backward_matches_autograd(n_base, N, L, p):
    from xna_basecaller_b200._lib import Handle
    sd = bo.reference_state_dict(n_base=n_base, seed=12, **REF_SCALE)
    x = synthetic_signal(41, N, L)
    T, seed = L // 5, 0x5eed0000 + N
    ps = [p] * 7
    cot = torch.randn(T, N, n_base ** 3 * (n_base + 1), generator=torch.Generator().manual_seed(9)) * 1e-2
    params = {k: v.clone().requires_grad_() for k, v in sd.items()}
    ref_scores = od.encoder_forward_dropout(params, x, n_base, ps, seed)
    ref_scores.backward(cot)
    ref = {k: q.grad for k, q in params.items()}
    h = Handle(ALPHABETS[n_base], 3, max_N=N, max_T=T, train=True)
    h.load_weights(sd)
    scores = h.encoder_train(x.cuda(), dropout_p=ps, seed=seed)
    err = (scores.cpu() - ref_scores.detach()).abs().max().item()
    assert err < 1e-2, err
    got = h.encoder_backward(cot.cuda())
    torch.cuda.synchronize()
    worst = _compare(got, ref)
    for k, (rel, cos) in sorted(worst.items()):
        print('%-32s rel %.4f  cos %.6f' % (k, rel, cos))
    for k, (rel, cos) in worst.items():
        assert rel <= REL_TOL and cos >= COS_TOL, (k, rel, cos)
    # the masks matter: the same step without dropout is far from this oracle
    plain = h.encoder_train(x.cuda())
    assert (plain.cpu() - ref_scores.detach()).abs().max().item() > 10 * max(err, 1e-3)
    h.close()


# ---------------------------------------------------------------------------------------------------------- seeding
def test_seeding_and_grad_accumulation():
    sd = bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE)
    _, model = _pair(sd, drop_rate_bottom=0.1)
    model.train()
    x = synthetic_signal(51, 16, 500)
    tg, tl = synthetic_targets(7, 16, 5, 40, 60)

    def step(split):
        model.zero_grad()
        for xc, tc, lc in zip(x.chunk(split), tg.chunk(split), tl.chunk(split)):
            scores = model(xc.cuda())
            loss = model.seqdist.ctc_loss(scores.float(), tc.cuda(), lc.cuda()) / split
            loss.backward()
        torch.cuda.synchronize()
        return scores.detach(), _named_grads(model)

    torch.manual_seed(1234)
    s1, g1 = step(1)
    torch.manual_seed(1234)
    s2, g2 = step(1)
    assert torch.equal(s1, s2)
    _assert_same_grads(g1, g2)
    s3, _ = step(1)                                   # the next forward draws a new seed: other masks
    assert not torch.equal(s1, s3)

    # grad_accum_split = 2 (Trainer.train_one_step): two forwards, each followed by its own backward
    torch.manual_seed(99)
    _, got = step(2)
    torch.manual_seed(99)
    seeds = [int(torch.empty((), dtype=torch.int64).random_().item()) for _ in range(2)]
    params = {k: v.clone().requires_grad_() for k, v in sd.items()}
    crf = bo.CRF(3, ALPHABETS[5])
    for xc, tc, lc, seed in zip(x.chunk(2), tg.chunk(2), tl.chunk(2), seeds):
        (crf.ctc_loss(od.encoder_forward_dropout(params, xc, 5, [0.1] * 7, seed), tc, lc) / 2).backward()
    names = [k for k in sd if not k.endswith('bias_hh_l0')]
    assert len(names) == len(got)
    for k, (n, g) in zip(names, got):
        assert n.rsplit('.', 2)[-2:] == k.rsplit('.', 2)[-2:]
        a, b = g.double().cpu().flatten(), params[k].grad.double().flatten()
        rel = ((a - b).norm() / b.norm().clamp_min(1e-30)).item()
        assert rel <= 5e-2, (k, rel)                  # the bound of test_trainer_train_one_step_through_the_plugin


def test_trainer_with_drop_rate_bottom_lowers_the_loss():
    from xna_basecaller_b200.training import Trainer
    _, model = _pair(bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE), drop_rate_bottom=0.1)
    N, L = 8, 600
    x = synthetic_signal(51, N, L)
    tg, tl = synthetic_targets(7, N, 5, 40, 60)
    trainer = Trainer(model, 'cuda')
    trainer.init_optimizer(1e-3)
    torch.manual_seed(0)
    first = None
    for _ in range(6):
        losses, grad_norm = trainer.train_one_step((x, tg, tl))
        assert np.isfinite(losses['loss']) and np.isfinite(grad_norm) and grad_norm > 0
        first = losses['loss'] if first is None else first
    assert losses['loss'] < first
    print('loss %.4f -> %.4f in 6 steps with drop_rate_bottom 0.1, last grad norm %.3f' % (first, losses['loss'], grad_norm))
