"""CPU tests of dropout in the training step (rnn_encoder(drop_rate_bottom=...)): the numpy restatement of the mask
contract (oracle/dropout.py) against Random123's known answers and the binomial distribution, and the recognition of
Dropout modules by Serial._stem / Serial._training_layout."""
import numpy as np
import pytest
import torch

from oracle import dropout as od
from test_cpu_host import sup_config

ALPHABET = 'NACGTX'


# Random123's known-answer vectors for philox4x32_10 (kat_vectors)
@pytest.mark.parametrize('ctr,key,want', [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    got = od.philox4x32_10(np.array(ctr, dtype=np.uint64), key)
    assert tuple(int(v) for v in got) == want


@pytest.mark.parametrize('p', [0.05, 0.5])
@pytest.mark.parametrize('site', [0, 4])
def test_keep_fraction_is_binomial(p, site):
    n = 10 ** 6
    k = od.keep(0x0123456789abcdef, site, p, n)
    sigma = np.sqrt(n * p * (1 - p))
    assert abs(int(k.sum()) - n * (1 - p)) <= 6 * sigma


def test_mask_contract_details():
    # element e takes word e & 3 of the call at counter e >> 2: a prefix is the start of a longer draw
    assert np.array_equal(od.keep(7, 2, 0.3, 13), od.keep(7, 2, 0.3, 1000)[:13])
    # sites and seeds (both key words) draw independent masks
    a = od.keep(7, 2, 0.5, 4096)
    assert not np.array_equal(a, od.keep(7, 3, 0.5, 4096))
    assert not np.array_equal(a, od.keep(7 + (1 << 32), 2, 0.5, 4096))
    assert od.keep(7, 2, 0.0, 4096).all()
    assert od.threshold(0.5) == (1 << 31, np.float32(2.0))
    assert od.threshold(0.0) == (0, np.float32(1.0))
    m = od.mask(5, 1, 0.25, (3, 16, 40)).numpy()
    assert set(np.unique(m).tolist()) <= {0.0, float(np.float32(1 / 0.75))}
    for bad in (-0.1, 1.0, 1.5, float('nan')):
        with pytest.raises(ValueError):
            od.threshold(bad)


def test_dropout_probabilities_are_checked():
    from xna_basecaller_b200 import _lib
    assert _lib.dropout_probabilities([0.1] * 7) == [0.1] * 7
    for bad in ([0.1] * 6, [0.1] * 6 + [1.0], [0.1] * 6 + [-0.5], [0.1] * 6 + [float('nan')], [0.1] * 6 + [1 - 1e-9]):
        with pytest.raises(ValueError):
            _lib.dropout_probabilities(bad)


def _model(**encoder):
    from xna_basecaller_b200 import util
    cfg = sup_config(ALPHABET)
    cfg['encoder'].update(encoder)
    return util.load_symbol(cfg, 'Model')(cfg)


def test_drop_rate_bottom_model_is_recognised():
    m = _model(drop_rate_bottom=0.1)
    enc = m.encoder
    assert sum(isinstance(x, torch.nn.Dropout) for x in enc) == 7
    stem = enc._stem()
    assert stem is not None and [c.conv.out_channels for c in stem] == [4, 16, 768]
    assert enc._stem_end() == 7                      # conv, drop, conv, drop, conv, drop, permute
    m.train()
    layout = enc._training_layout()
    assert layout is not None
    _, lstms, head, p = layout
    assert len(lstms) == 5 and p == [0.1] * 7
    m.eval()                                         # Dropout modules in eval mode drop nothing
    assert enc._training_layout()[3] == [0.0] * 7
    plain = _model()
    plain.train()
    assert plain.encoder._stem_end() == 4 and plain.encoder._training_layout()[3] == [0.0] * 7


def test_single_sites_and_misplaced_dropout():
    from xna_basecaller_b200.nn import Serial
    m = _model(drop_rate_bottom=0.2)
    m.train()
    mods = list(m.encoder)
    drops = [i for i, x in enumerate(mods) if isinstance(x, torch.nn.Dropout)]
    # each site is optional: keep only one Dropout at a time
    for site, keep in enumerate(drops):
        sub = Serial([x for i, x in enumerate(mods) if i not in drops or i == keep])
        sub.train()
        p = sub._training_layout()[3]
        assert p == [0.2 if s == site else 0.0 for s in range(7)]
    permute = next(i for i, x in enumerate(mods) if x.__class__.__name__ == 'Permute')
    for pos in (0, permute + 1, len(mods) - 1, len(mods), drops[3] + 1):
        # before conv1, after the Permute, after LSTM 4, after the head, and a second Dropout right after another
        bad = Serial(mods[:pos] + [torch.nn.Dropout(0.1)] + mods[pos:])
        bad.train()
        assert bad._training_layout() is None, pos
        ok = Serial(mods[:pos] + [torch.nn.Dropout(0.0)] + mods[pos:])     # p = 0 is the identity wherever it stands
        ok.train()
        assert ok._training_layout() is not None, pos
    # the inference stem skips Dropouts, even one in front of it
    assert Serial([torch.nn.Dropout(0.1)] + mods)._stem() is not None


def test_training_with_head_dropout_raises():
    """LinearCRFEncoder(drop_rate > 0): the forward placement of the head's dropout is not recorded here, so training
    refuses instead of silently training without it.  The check runs before anything reaches the device."""
    m = _model(drop_rate_bottom=0.1, drop_rate=0.1)
    m.train()
    with pytest.raises(RuntimeError, match='drop_rate'):
        m(torch.zeros(8, 1, 500))
    m.encoder[-1].dropout.p = 0.0
    assert m.encoder._training_layout() is not None
