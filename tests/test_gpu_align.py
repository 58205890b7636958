"""Validation accuracy on the GPU: xb_align_counts against the C checker (oracle/c/align_exact.c) integer for integer,
util.accuracy on known answers, and Trainer.validate_one_step / validate_one_epoch against the decode, decode_ref, the
checker and ctc_loss."""
import types

import numpy as np
import pytest
import torch

from make_golden import ALPHABETS, synthetic_signal
from oracle import bonito_oracle as bo
from oracle import align_exact
from test_cpu_align import KNOWN, _mutate

pytestmark = pytest.mark.gpu

LETTERS = 'ACGTX'


def _rand(rs, n, abc=LETTERS):
    return ''.join(abc[k] for k in rs.randint(len(abc), size=n))


def _kernel_vs_checker(seqs, refs, seq_width=None, ref_width=None, pad=0):
    """Rows of the given widths (plus `pad` unused bytes per row, passed as a column slice so that the row stride exceeds
    the row width) through xb_align_counts and through the checker."""
    from xna_basecaller_b200._lib import align_counts
    s, sl = align_exact.rows(seqs, seq_width)
    r, rl = align_exact.rows(refs, ref_width)
    want = align_exact.align_counts(s, sl, r, rl, threads=8)
    s_dev = torch.from_numpy(np.pad(s, ((0, 0), (0, pad)), constant_values=7)).cuda()[:, :s.shape[1]]
    r_dev = torch.from_numpy(np.pad(r, ((0, 0), (0, pad)), constant_values=7)).cuda()[:, :r.shape[1]]
    got = align_counts(s_dev, torch.from_numpy(sl).cuda(), r_dev, torch.from_numpy(rl).cuda()).cpu().numpy()
    bad = np.nonzero((got != want).any(1))[0]
    assert len(bad) == 0, [(int(p), len(seqs[p]), len(refs[p]), got[p].tolist(), want[p].tolist()) for p in bad[:5]]
    return got


def test_align_counts_realistic_batch():
    """512 pairs, decodes up to T = 800, references up to 600: mutated copies (10 / 30 % substitutions, insertions,
    deletions), pieces of the decode, unrelated sequences."""
    rs = np.random.RandomState(21)
    seqs, refs = [], []
    for k in range(512):
        seq = _rand(rs, rs.randint(1, 801))
        kind = k % 4
        if kind in (0, 1):
            ref = _mutate(rs, seq, 0.1 if kind == 0 else 0.3, LETTERS)
        elif kind == 2:
            a = rs.randint(len(seq))
            ref = _mutate(rs, seq[a:a + rs.randint(1, 600)], 0.1, LETTERS)
        else:
            ref = _rand(rs, rs.randint(0, 601))
        seqs.append(seq)
        refs.append(ref[:600])
    got = _kernel_vs_checker(seqs, refs, 800, 600)
    assert (got[:, 0] > 0).mean() > 0.9


def test_align_counts_edge_cases():
    """Empty and single-letter sides, seq longer and shorter than ref, references across band boundaries (512 columns per
    band) and far beyond one band, both lengths at the 32767 limit (against a short partner), 13 pairs (not a multiple
    of the 4 pairs per CTA) and row strides larger than the rows."""
    rs = np.random.RandomState(8)
    long_seq = _rand(rs, 32767)
    long_ref = _rand(rs, 32767)
    mid = _rand(rs, 1600)
    pairs = [
        ('', 'ACGT'), ('ACGT', ''), ('', ''), ('A', 'A'), ('A', 'C'), ('A', 'AAAAAAA'), ('TTTTTTT', 'T'),
        (mid[400:700], mid),                                   # seq shorter than ref, match inside band 0
        (_mutate(rs, mid[480:560], 0.1, LETTERS), mid[:1024]),  # match across the first band boundary
        (mid, _mutate(rs, mid[1000:1100], 0.1, LETTERS)),       # seq longer than ref
        (_mutate(rs, mid, 0.1, LETTERS), mid),                  # both long, 4 bands
        (_mutate(rs, long_seq[20000:20050], 0.1, LETTERS) + 'A' * 5, long_seq[20000:20060]),
        (long_seq, _mutate(rs, long_seq[30000:30060], 0.1, LETTERS)),
        (_mutate(rs, long_ref[32700:], 0.1, LETTERS), long_ref),  # 64 bands, match in the last
        (long_ref[511:541], long_ref),                           # match starting on a band's last column
    ]
    seqs, refs = [p[0] for p in pairs], [p[1] for p in pairs]
    assert len(seqs) % 4 != 0
    assert max(map(len, seqs)) == 32767 and max(map(len, refs)) == 32767
    got = _kernel_vs_checker(seqs, refs, pad=5)
    assert got[3].tolist() == [5, 1, 0, 0, 0] and got[2].tolist() == [0] * 5
    # the same pairs with wider rows
    _kernel_vs_checker(seqs[:11], refs[:11], 33000, 33000)


def test_align_counts_rejects_bad_lengths():
    from xna_basecaller_b200._lib import align_counts
    rows = torch.zeros(2, 40000, dtype=torch.int8, device='cuda')
    ok = torch.tensor([10, 10], dtype=torch.int32, device='cuda')
    for bad in ([10, 32768], [-1, 10], [10, 40001]):
        with pytest.raises(RuntimeError, match=r'xb_align_counts failed \(-1\)'):
            align_counts(rows, torch.tensor(bad, dtype=torch.int32, device='cuda'), rows, ok)
    with pytest.raises(RuntimeError, match=r'\(-1\)'):                 # longer than the row stride (5 bytes)
        align_counts(torch.zeros(2, 5, dtype=torch.int8, device='cuda'), ok, rows, ok)
    assert align_counts(rows, ok, rows, ok).cpu().tolist() == [[50, 10, 0, 0, 0]] * 2   # any byte is a letter


def test_util_accuracy_known_answers():
    from xna_basecaller_b200 import util
    for seq, ref, _, acc_half, acc_zero, acc_bal in KNOWN:
        assert util.accuracy(ref, seq, min_coverage=0.5) == pytest.approx(acc_half, abs=1e-12)
        assert util.accuracy(ref, seq) == pytest.approx(acc_zero, abs=1e-12)
        assert util.accuracy(ref, seq, balanced=True) == pytest.approx(acc_bal, abs=1e-12)
    assert util.accuracy('ACGT', '') == 0.0 and util.accuracy('', 'ACGT') == 0.0


def _golden_model():
    from xna_basecaller_b200 import util
    cfg = {'global_norm': {'state_len': 3}, 'input': {'features': 1}, 'labels': {'labels': ALPHABETS[5]},
           'model': {'package': 'xna_basecaller_b200.crf'},
           'encoder': {'stride': 5, 'activation': 'swish', 'features': 768, 'winlen': 19, 'scale': 5.0,
                       'rnn_type': 'lstm', 'blank_score': 2.0}}
    model = util.load_symbol(cfg, 'Model')(cfg)
    model.load_state_dict(bo.reference_state_dict(n_base=5, seed=3))      # amplified head: decodes mix blanks and moves
    return model.cuda()


def _mutated_targets(model, x, seed):
    """Targets = the model's own decodes mutated (~10 %), as 1-based labels; an empty decode gets a random target."""
    model.eval()
    with torch.no_grad():
        decodes = model.decode_batch(model(x.cuda()).float())
    rs = np.random.RandomState(seed)
    refs = [_mutate(rs, d, 0.1, LETTERS) if d else _rand(rs, 20) for d in decodes]
    refs = [r if r else 'A' for r in refs]
    tg = np.zeros((len(refs), max(map(len, refs)) + 3), dtype=np.int64)
    for i, r in enumerate(refs):
        tg[i, :len(r)] = ['NACGTX'.index(c) for c in r]
    return torch.from_numpy(tg), torch.tensor([len(r) for r in refs], dtype=torch.int64), decodes


def test_validate_one_step_matches_its_parts():
    from xna_basecaller_b200 import util
    from xna_basecaller_b200.training import Trainer
    model = _golden_model()
    x = synthetic_signal(71, 16, 1000)
    tg, tl, decodes = _mutated_targets(model, x, 4)
    assert sum(map(len, decodes)) > 16 * 20
    trainer = Trainer(model, 'cuda')
    seqs, refs, accs, loss = trainer.validate_one_step((x, tg, tl))
    with torch.no_grad():
        scores = model(x.cuda()).float()
        want_loss = model.seqdist.ctc_loss(scores, tg.cuda(), tl.cuda()).item()
    assert seqs == model.decode_batch(scores) == decodes
    assert refs == [util.decode_ref(t, model.alphabet) for t in tg]
    counts = align_exact.align_strings(seqs, refs)
    assert accs == [util._accuracy(c, len(r), False, 0.5) if len(s) else 0. for c, r, s in zip(counts, refs, seqs)]
    assert 50 < np.mean(accs) <= 100
    assert loss == pytest.approx(want_loss, rel=1e-6)


def test_validate_one_epoch_over_a_device_loader():
    from xna_basecaller_b200 import data
    from xna_basecaller_b200.training import Trainer
    model = _golden_model()
    x = synthetic_signal(72, 24, 1000)
    tg, tl, _ = _mutated_targets(model, x, 5)
    ds = types.SimpleNamespace(chunks=x.numpy(), targets=tg.numpy(), lengths=tl.numpy())
    loader = data.DeviceChunkLoader(ds, batch_size=8, device='cuda')
    trainer = Trainer(model, 'cuda', valid_loader=loader)
    loss, mean, median = trainer.validate_one_epoch()
    steps = [trainer.validate_one_step(b) for b in loader]
    accs = sum((s[2] for s in steps), [])
    assert len(accs) == 24
    assert loss == pytest.approx(np.mean([s[3] for s in steps]), rel=1e-12)
    assert mean == np.mean(accs) and median == np.median(accs)
    assert not model.training
