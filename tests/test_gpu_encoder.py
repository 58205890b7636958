"""GPU parity tests of the CUDA encoder (conv stem, LSTM stack, CRF head) against the fp32 oracle and the
golden vectors produced by the reference's own bonito.nn / bonito.crf.model code.

Tolerance (BASELINE.json north_star): max abs error <= 1e-2 on the CRF scores (range +-5) with 16-bit
tensor-core operands against the fp32 reference.  The 16-bit type is fp16 by default -- what the reference
itself runs on GPU (bonito/util.py:360-363); the bf16 option rounds the weights to bfloat16 and keeps fp16 activations
(tests/precision_attribution.py shows why), and meets the same bound."""
import numpy as np
import pytest
import torch

from make_golden import ALPHABETS, synthetic_signal
from oracle import bonito_oracle as bo

pytestmark = pytest.mark.gpu

SCORE_TOL_F16 = 1e-2          # reference-scale weights (unit gains, like the reference's own init)
SCORE_TOL_F16_AMPLIFIED = 6e-2  # test weights with a 12x head gain: fp16 weight rounding alone gives ~3e-2
SCORE_TOL_BF16 = 1e-2           # bf16-rounded weights x fp16 activations at reference scale


@pytest.fixture(scope='module')
def enc5():
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=16, max_T=400)
    sd = bo.reference_state_dict(n_base=5, seed=11)
    h.load_weights(sd)
    yield h, sd
    h.close()


@pytest.mark.parametrize('M,N,K', [(128, 128, 64), (256, 384, 768), (1000, 640, 320), (77, 128, 128)])
def test_gemm_selftest(M, N, K):
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=4, max_T=8, encoder=False)
    g = torch.Generator(device='cuda').manual_seed(M + N + K)
    A = torch.randn(M, K, device='cuda', generator=g).half()
    B = torch.randn(N, K, device='cuda', generator=g).half()
    D = h.gemm_selftest(A, B)
    ref = A.float() @ B.float().t()
    err = (D - ref).abs().max().item()
    assert err < 1e-2 * (K / 64) ** 0.5, err
    h.close()


def test_conv_stem(enc5, golden):
    h, sd = enc5
    x = synthetic_signal(21, 2, 500)
    got = h.conv_stem(x.cuda()).float().cpu()             # (T, N, 768)
    ref = bo.conv_stem(sd, x).permute(2, 0, 1)
    err = (got - ref).abs()
    assert (err / (1 + ref.abs())).max().item() < 4e-3
    gold = torch.from_numpy(golden['encoder']['n5_stem_sub'])       # reference code output (N, 48, T)
    assert ((got.permute(1, 2, 0)[:, ::16, :] - gold).abs() / (1 + gold.abs())).max().item() < 4e-3


@pytest.mark.parametrize('N,L', [(3, 100), (5, 165), (2, 2000), (9, 1280)])
def test_conv_stem_shapes(enc5, N, L):
    """conv3_gemm.cu: row blocks that cross chunk edges (T not a multiple of 32: row-copy path), chunks shorter than a
    block (T = 20), T = 800 / 256 (TMA-store path only), a last row tile that is mostly padding."""
    h, sd = enc5
    x = synthetic_signal(100 + N, N, L)
    got = h.conv_stem(x.cuda()).float().cpu()
    ref = bo.conv_stem(sd, x).permute(2, 0, 1)
    assert got.shape == ref.shape
    assert ((got - ref).abs() / (1 + ref.abs())).max().item() < 4e-3


@pytest.mark.parametrize('reverse', [True, False])
def test_lstm_layer(enc5, reverse):
    h, sd = enc5
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(60, 5, 768, generator=g) * 0.5).half()
    p = 'encoder.4.rnn.'
    ref = bo.lstm_layer(x.float(), sd[p + 'weight_ih_l0'], sd[p + 'weight_hh_l0'], sd[p + 'bias_ih_l0'],
                        sd[p + 'bias_hh_l0'], reverse)
    got = h.lstm(0, x.cuda(), reverse).float().cpu()
    assert (got - ref).abs().max().item() < 4e-3


@pytest.mark.parametrize('N,T', [(100, 24), (200, 17), (577, 6)])
def test_lstm_layer_multi_group(N, T):
    """Several batch groups per launch (96 chunks each), uneven last group, and more than one launch (N > 576)."""
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=N, max_T=T)
    sd = bo.reference_state_dict(n_base=5, seed=11)
    h.load_weights(sd)
    g = torch.Generator().manual_seed(N + T)
    x = (torch.randn(T, N, 768, generator=g) * 0.5).half()
    p = 'encoder.5.rnn.'
    for reverse in (False, True):
        ref = bo.lstm_layer(x.float(), sd[p + 'weight_ih_l0'], sd[p + 'weight_hh_l0'], sd[p + 'bias_ih_l0'],
                            sd[p + 'bias_hh_l0'], reverse)
        got = h.lstm(1, x.cuda(), reverse).float().cpu()
        assert (got - ref).abs().max().item() < 4e-3
    h.close()


def test_lstm_first_layer_golden(enc5, golden):
    """encoder.4 of the reference Model on the reference stem output."""
    h, sd = enc5
    x = synthetic_signal(21, 2, 500)
    stem = h.conv_stem(x.cuda())
    got = h.lstm(0, stem, True).float().cpu()
    gold = torch.from_numpy(golden['encoder']['n5_lstm1_sub'])      # (T, N, 48)
    assert (got[:, :, ::16] - gold).abs().max().item() < 5e-3


def test_crf_head(enc5):
    h, sd = enc5
    g = torch.Generator().manual_seed(6)
    x = (torch.rand(50, 3, 768, generator=g) * 2 - 1).half()
    ref = bo.crf_head(sd, x.float(), 5)
    got = h.crf_head(x.cuda()).cpu()
    assert got.shape == ref.shape
    assert torch.equal(got.view(50, 3, 125, 6)[..., 0], torch.full((50, 3, 125), 2.0))
    # against the fp32 head: bounded by the fp16 rounding of the (12x amplified) head weights
    assert (got - ref).abs().max().item() < SCORE_TOL_F16_AMPLIFIED
    # against the same head evaluated on fp16-rounded weights: only accumulation order / tanh differ
    sdq = dict(sd)
    sdq['encoder.9.linear.weight'] = sd['encoder.9.linear.weight'].half().float()
    assert (got - bo.crf_head(sdq, x.float(), 5)).abs().max().item() < 1e-3


@pytest.mark.parametrize('n_base', [5, 6])
def test_encoder_scores_vs_reference_golden(golden, n_base):
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[n_base], 3, max_N=8, max_T=200)
    sd = bo.reference_state_dict(n_base=n_base, seed=11)
    h.load_weights(sd)
    x = synthetic_signal(21, 2, 500)
    got = h.encoder(x.cuda()).cpu()
    gold = torch.from_numpy(golden['encoder']['n%d_scores' % n_base])
    assert got.shape == gold.shape
    err = (got - gold).abs().max().item()
    assert err <= SCORE_TOL_F16_AMPLIFIED, err
    # decoded strings from the CUDA scores equal the reference's decode of its own fp32 scores
    seq, _, lens = h.decode(got, want_qstring=False)
    strings = [bytes(seq[i, :lens[i]].cpu().numpy().astype('u1')).decode() for i in range(2)]
    assert strings == list(golden['encoder']['n%d_strings' % n_base])
    h.close()


def test_encoder_scores_reference_scale_tolerance(golden):
    """The north-star tolerance: max abs error <= 1e-2 on the scores against the reference's fp32 output."""
    from make_golden import REF_SCALE
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=8, max_T=200)
    h.load_weights(bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE))
    got = h.encoder(synthetic_signal(23, 2, 500).cuda()).cpu()
    err = (got - torch.from_numpy(golden['encoder']['r5_scores'])).abs().max().item()
    print('fp16 max abs score error at reference scale', err)
    assert err <= SCORE_TOL_F16, err
    h.close()


def test_encoder_bf16_option():
    from make_golden import REF_SCALE
    from xna_basecaller_b200._lib import Handle
    h = Handle(ALPHABETS[5], 3, max_N=8, max_T=200, bf16=True)
    sd = bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE)
    h.load_weights(sd)
    x = synthetic_signal(22, 3, 500)
    got = h.encoder(x.cuda()).cpu()
    ref = bo.encoder_forward(sd, x, 5)
    err = (got - ref).abs().max().item()
    print('bf16 max abs score error', err)
    assert err <= SCORE_TOL_BF16, err
    h.close()


def test_head_exp_mode_and_fused_route(enc5):
    """The CRF head's exp epilogue writes exactly xb_score_exp(score) (blank column included), and the fused
    xb_basecall_chunks route (head -> exp(scores) -> linear-domain decode) returns the packed rows of the two-call route."""
    from oracle import cexact
    h, sd = enc5
    g = torch.Generator().manual_seed(8)
    x = (torch.rand(70, 5, 768, generator=g) * 2 - 1).half().cuda()
    s = h.crf_head(x)
    e = h.crf_head(x, exp=True)
    assert np.array_equal(e.cpu().numpy().view(np.uint32), cexact.score_exp(s.cpu().numpy()).view(np.uint32))
    sig = synthetic_signal(27, 6, 1500)
    seq, _, lens = h.basecall_chunks(sig.cuda())
    seq2, _, lens2 = h.decode(h.encoder(sig.cuda()), want_qstring=False)
    assert torch.equal(seq, seq2) and torch.equal(lens, lens2)
    assert int(lens.sum()) > 0


def test_compute_scores_host_end_to_end(enc5, golden):
    """H2D -> encoder -> decode -> D2H through the host-buffer entry point, against the reference's
    compute_scores output (left-packed int8 rows)."""
    h, sd = enc5
    x = synthetic_signal(21, 2, 500)
    seq, lens = h.compute_scores_host(x[:, 0, :].contiguous().pin_memory())
    gold = golden['encoder']['n5_cs_sequence']
    assert np.array_equal(seq.numpy(), gold)
    assert lens.tolist() == [(gold[i] != 0).sum() for i in range(2)]
    assert h.launches > 0


def test_training_forward_loss_config5():
    """BASELINE config 5 (forward half): encoder forward in bf16 + CTC-CRF loss on spliced-UB targets, full
    chunk length; checked against the fp32 oracle on two chunks of the batch (chunks are independent)."""
    from make_golden import REF_SCALE
    from xna_basecaller_b200._lib import Handle
    N, L = 96, 4000
    h = Handle(ALPHABETS[5], 3, max_N=N, max_T=L // 5, bf16=True)
    sd = bo.reference_state_dict(n_base=5, seed=12, **REF_SCALE)
    h.load_weights(sd)
    x = synthetic_signal(31, N, L)
    rs = np.random.RandomState(3)
    lengths = rs.randint(350, 451, size=N)
    tg = np.zeros((N, 450), dtype=np.int64)
    for i, n in enumerate(lengths):
        tg[i, :n] = rs.randint(1, 5, size=n)
        pos = 3
        while pos < n - 3:                       # UB label (5) at ~9 % of positions, at least 5 bases apart
            if rs.rand() < 0.45:
                tg[i, pos] = 5
            pos += 5
    tg, tl = torch.from_numpy(tg), torch.from_numpy(lengths.astype(np.int64))
    scores = h.encoder(x.cuda())
    loss = h.ctc_loss(scores, tg, tl).cpu()
    assert loss.shape == (N,) and torch.isfinite(loss).all() and (loss > 0).all()
    pick = [0, N - 1]
    ref_scores = bo.encoder_forward(sd, x[pick], 5)
    ref = bo.CRF(3, ALPHABETS[5]).ctc_loss(ref_scores, tg[pick], tl[pick], reduction='none')
    # same loss from the CUDA scores through the oracle (isolates the loss kernel), then end to end in bf16
    same = bo.CRF(3, ALPHABETS[5]).ctc_loss(scores[:, pick].cpu(), tg[pick], tl[pick], reduction='none')
    np.testing.assert_allclose(loss[pick].numpy(), same.numpy(), rtol=5e-5)
    np.testing.assert_allclose(loss[pick].numpy(), ref.numpy(), rtol=3e-2)
    h.close()


def test_batch_position_independence_odd_sizes():
    """A chunk's scores and decode do not depend on where it sits in the batch or on the batch size: batches of odd sizes
    (uneven LSTM groups and sub-batches, partial GEMM tiles, a second recurrence launch at N > 576) built by repeating five
    chunks give, for every copy, the bits of the five-chunk batch."""
    from xna_basecaller_b200._lib import Handle
    T, L = 120, 600
    h = Handle(ALPHABETS[5], 3, max_N=1000, max_T=T)
    h.load_weights(bo.reference_state_dict(n_base=5, seed=11))
    base = synthetic_signal(33, 5, L)[:, 0, :].contiguous().cuda()
    s0 = h.encoder(base)
    seq0, _, lens0 = h.decode(s0, want_qstring=False)
    for N in (1, 7, 97, 300, 577, 1000):
        idx = torch.arange(N, device='cuda') % 5
        s = h.encoder(base[idx].contiguous())
        assert torch.equal(s, s0[:, idx]), N
        seq, _, lens = h.decode(s, want_qstring=False)
        assert torch.equal(seq, seq0[idx]) and torch.equal(lens, lens0[idx]), N
    h.close()


def test_pipelined_host_entry_points_match_the_blocking_one(enc5):
    """xb_compute_scores_submit / _wait over five different batches in two slots == xb_basecall_chunks on device copies of
    the same batches."""
    h, _ = enc5
    batches = [synthetic_signal(40 + i, 3, 500)[:, 0, :].contiguous().pin_memory() for i in range(5)]
    want = []
    for b in batches:
        seq, _, lens = h.basecall_chunks(b.cuda())
        want.append((seq.cpu(), lens.cpu()))
    seqs = [torch.empty(3, 100, dtype=torch.int8).pin_memory() for _ in range(2)]
    lens = [torch.empty(3, dtype=torch.int32).pin_memory() for _ in range(2)]
    got = []
    for i, b in enumerate(batches):
        if i >= 2:
            h.compute_scores_wait(i & 1)
            got.append((seqs[i & 1].clone(), lens[i & 1].clone()))
        h.compute_scores_submit(i & 1, b, seqs[i & 1], lens[i & 1])
    for i in (3, 4):
        h.compute_scores_wait(i & 1)
        got.append((seqs[i & 1].clone(), lens[i & 1].clone()))
    assert len(got) == 5
    for (ws, wl), (gs, gl) in zip(want, got):
        assert torch.equal(ws, gs) and torch.equal(wl, gl)
    assert any(int(wl.sum()) > 0 for _, wl in want)
