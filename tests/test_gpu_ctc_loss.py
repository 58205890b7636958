"""The CTC-CRF loss and its gradient w.r.t. the scores (xb_ctc_crf_loss_fwd / _bwd: ctc_simple_kernel and
ctc_simple_bwd_kernel, with the full-lattice posteriors of xb_decode_lin and logZ of xb_decode_alpha) against the float64
reference oracle/train_stages.ctc_loss_backward, at the training shape and at the kernels' edges:

  * the training distribution (T = 800, targets of 350 to 450 bases with X spliced in as bench.py's training step does)
    for n_base 4, 5 and 6, with and without normalise, and upstream gradients of 0, < 0 and 1/N;
  * the benchmark's shape, N = 512, with the benchmark's own targets, and a sequence's result at any batch position;
  * block sizes: npos = Lmax - 2 in {1, 31, 32, 33, 383, 385, 1024} (one position; one inactive lane at 31 and 383;
    whole warps at 32; one active lane in the last warp at 33 and 385; the largest block), and on both sides of the backward's switch to
    ceil(S / 128) * 32 threads for its score row (npos 64/65, 160/161, 352/353 for n_base 4, 5, 6); Lmax = 1027 and
    Lmax = 2 are refused before anything is launched;
  * time edges (T = 1, 2, and a target of T + 3 bases, which has exactly one alignment);
  * colliding numerator edges (homopolymers and 2-base repeats), padding and garbage after a target's length, and targets
    no alignment reaches;
  * the plugin route, CTC_CRF.ctc_loss, with fp32 and fp16 scores and loss_clip.

Every comparison is per sequence, so that no sequence's error hides behind a larger gradient in another row.  Loss:
relative error.  Gradient: relative error in the 2-norm, 1 - cosine, and the max abs error in units of |grad_loss| / len,
the factor by which the kernel scales the sequence's posteriors (so an error in posterior units).

Two launches of the backward on the same sequence need not agree bit for bit: each step adds the numerator of every
target position to its edge with a shared-memory atomicAdd, in no fixed order.  fp32 addition is commutative, so an edge
that receives at most two non-zero terms in a step gets the same sum in any order; three or more can round differently.
A sequence in which no stay edge (state) and no move edge (state and the base it dropped) is shared by three positions
must therefore be repeated bit for bit; any other agrees within ATOMIC_REL.  _check_same says which case applies.

The kernels work in fp32 in the log domain.  Their error against float64 grows with the magnitude of the alignment
lattice's alpha and beta, accumulated over T steps.  With normalise every score is lowered by logZ / T, and on these
random scores alpha ends near -(loss * len), up to ~-5e3 at T = 1030, where one ulp is 4.9e-4: posteriors come out ~1e-2
off.  Without normalise the same batches agree ~10x closer.  Hence four sets of bounds, each a 2-4x multiple of the
largest error observed in its cases:

Largest errors observed on a B200 (1000 W power limit), per sequence, and the bounds:
                                     loss rel       grad rel       max abs / scale   1 - cos
  RAW   normalise=False, every T     1.5e-6  5e-6   2.4e-3  7e-3   3.3e-3  7e-3      6.7e-7  2e-6
  NORM  normalise=True, T <= 800     7.0e-6  2e-5   6.7e-3  2e-2   1.0e-2  3e-2      5.7e-6  2e-5
  NORM_LONG        T = 1030, full    1.2e-5  4e-5   1.4e-2  4e-2   1.6e-2  4e-2      4.4e-5  1.3e-4
  NORM_LONG_SHORT  T = 1030, short   1.4e-5  4e-5   2.2e-2  5e-2   2.8e-2  7e-2      4.6e-5  1.5e-4
("full": targets of Lmax and Lmax - 1 bases; "short": Lmax // 4 and 3 bases.)  test_gpu_crf.py bounds the gradient
against the fp32 oracle at 2e-5 absolute for 350..450-base targets and |grad_loss| <= 1, 8e-3 in these units for a
400-base target at grad_loss 1.  RAW is within that.  NORM is not: against float64, n_base 6 homopolymers with normalise
reach 1.0e-2, which is fp32 rounding of log-domain sums of that size, not a kernel fault; rescaled recursions would be
needed to go lower.
Repeated launches (_check_same): at most 1.0e-8 relative where the atomics' order applies, against ATOMIC_REL 1e-6.
"""
import numpy as np
import pytest
import torch

from make_golden import ALPHABETS
from oracle import bonito_oracle as bo
from oracle import train_stages as ts

pytestmark = pytest.mark.gpu

# bounds per sequence (see the table above): loss relative error; gradient relative 2-norm error, max abs error in units of
# |grad_loss| / len, and 1 - cosine
RAW = dict(loss=5e-6, rel=7e-3, abs=7e-3, cos=2e-6)              # normalise=False, every T
NORM = dict(loss=2e-5, rel=2e-2, abs=3e-2, cos=2e-5)             # normalise=True, T <= 800
NORM_LONG = dict(loss=4e-5, rel=4e-2, abs=4e-2, cos=1.3e-4)      # normalise=True, T = 1030, targets of Lmax - 1 and Lmax
NORM_LONG_SHORT = dict(loss=4e-5, rel=5e-2, abs=7e-2, cos=1.5e-4)  # normalise=True, T = 1030, targets of 3 .. Lmax // 4
ATOMIC_REL = 1e-6
MAX_T = 1030


@pytest.fixture(scope='module')
def handles():
    from xna_basecaller_b200._lib import Handle
    hs = {n: Handle(ALPHABETS[n], 3, max_N=512, max_T=MAX_T, encoder=False) for n in (4, 5, 6)}
    yield hs
    for h in hs.values():
        h.close()


def _scores(seed, T, N, n_base):
    """Non-blank scores ~U(-5, 5) and a constant blank 2, the range of the head's 5 tanh(.) (make_golden.synthetic_scores),
    drawn on the GPU."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    s = torch.rand(T, N, n_base ** 3, n_base + 1, generator=g, device='cuda') * 10 - 5
    s[..., 0] = 2.0
    return s.reshape(T, N, -1)


def _train_targets(seed, N, n_base, lo=350, hi=450):
    """bench.py's train_step_leg targets: ACGT drawn uniformly, and X (label 5) at 99 % of every 11th position from the
    5th.  With seed 3 and n_base 5 these are the benchmark's own.  n_base 6 puts X or Y there, n_base 4 has no X."""
    rs = np.random.RandomState(seed)
    lens = rs.randint(lo, hi + 1, N)
    tg = np.zeros((N, int(lens.max())), dtype=np.int64)
    for i, n in enumerate(lens):
        seq = rs.randint(1, 5, n)
        if n_base >= 5:
            cand = np.arange(5, n - 5, 11)
            sel = cand[rs.rand(len(cand)) < 0.99]
            seq[sel] = 5 if n_base == 5 else rs.randint(5, 7, len(sel))
        tg[i, :n] = seq
    return torch.from_numpy(tg), torch.from_numpy(lens)


def _pad(rows, width):
    tg = torch.zeros(len(rows), width, dtype=torch.int64)
    for i, r in enumerate(rows):
        tg[i, :len(r)] = torch.as_tensor(r)
    return tg, torch.tensor([len(r) for r in rows])


def _de_bruijn(k, n=3):
    """Labels 1..k in which every n-mer occurs once (a de Bruijn sequence, made linear): no two target positions share an
    edge."""
    a, seq = [0] * (k * n), []

    def db(t, p):
        if t > n:
            if n % p == 0:
                seq.extend(a[1:p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, k):
                a[t] = j
                db(t + 1, t)
    db(1, 1)
    return [v + 1 for v in seq + seq[:n - 1]]


def _check_loss(what, got, ref, b):
    rel = ((got.double() - ref) / ref).abs()
    n = int(rel.argmax())
    print('%-58s loss rel %.2e (seq %d)  (bound %.1e)' % (what, rel[n], n, b['loss']))
    assert rel[n] <= b['loss'], (what, n, rel[n].item())


def _check(what, got, ref, gl, tl, b):
    """Gradients (T, N, S), one sequence at a time: the relative error in the 2-norm, 1 - cosine, and the max abs error in
    units of |grad_loss| / len, the factor the kernel scales the sequence's posteriors by.  Each sequence is held to the
    bounds on its own, so a large gradient in one row cannot hide an error in another.  A sequence whose reference
    gradient is zero (grad_loss 0, or no numerator and no normalise) must be exactly zero."""
    x, y = got.double(), ref.to(got.device)
    d = x - y
    xn, yn = x.norm(dim=(0, 2)), y.norm(dim=(0, 2))
    zero = (yn == 0).cpu()
    assert not got[:, zero.to(got.device)].any(), (what, torch.nonzero(zero).flatten().tolist())
    rel = (d.norm(dim=(0, 2)) / yn)[~zero.to(got.device)].cpu()
    cos1 = (1 - (x * y).sum((0, 2)) / (xn * yn))[~zero.to(got.device)].cpu()
    scale = (gl.double().abs() / tl.double()).to(got.device)
    mab = (d.abs().amax(dim=(0, 2)) / scale)[~zero.to(got.device)].cpu()
    ids = torch.nonzero(~zero).flatten()
    worst = [(v.max().item(), int(ids[v.argmax()])) for v in (rel, mab, cos1)]
    print('%-58s grad rel %.2e (seq %d)  max abs / scale %.2e (seq %d)  1 - cos %.2e (seq %d)  (bounds %.0e, %.0e, %.0e)'
          % (what, *worst[0], *worst[1], *worst[2], b['rel'], b['abs'], b['cos']))
    assert worst[0][0] <= b['rel'] and worst[1][0] <= b['abs'] and worst[2][0] <= b['cos'], (what, worst)


def _compare(what, h, n_base, s, tg, tl, gl, normalise=True, b=None):
    """Kernel loss and gradient against the float64 reference, bounds b (default NORM or RAW); returns the kernel's
    (loss, grad)."""
    b = b or (NORM if normalise else RAW)
    loss = h.ctc_loss(s, tg, tl, normalise=normalise)
    grad = h.ctc_loss_bwd(s, tg, tl, gl, normalise=normalise)
    rl, rg = ts.ctc_loss_backward(s, tg, tl, gl, n_base, normalise=normalise)
    what = '%s, normalise=%d' % (what, normalise)
    _check_loss(what, loss, rl, b)
    _check(what, grad, rg, gl, tl, b)
    for n in torch.nonzero(gl == 0).flatten().tolist():
        assert not grad[:, n].any(), (what, n)
    return loss, grad


def _shared(tg, tl, T):
    """Per sequence, the most target positions whose numerator lands on one edge: positions with the same state (stay
    edge) or the same state and dropped base (move edge).  0 for a target no alignment reaches."""
    out = []
    for row, n in zip(tg.tolist(), tl.tolist()):
        if n < 3 or n > len(row) or n - 3 > T:
            out.append(0)
            continue
        r = [max(v - 1, 0) for v in row[:n]]
        stay = {}
        for j in range(n - 2):
            stay[tuple(r[j:j + 3])] = stay.get(tuple(r[j:j + 3]), 0) + 1
        move = {}
        for j in range(1, n - 2):
            move[tuple(r[j - 1:j + 3])] = move.get(tuple(r[j - 1:j + 3]), 0) + 1
        out.append(max(list(stay.values()) + list(move.values())))
    return torch.tensor(out)


def _check_same(what, got, ref, tg, tl, T):
    """Two launches' gradients of the same sequences (T, N, S): bit for bit where no edge takes three numerator terms in a
    step, within ATOMIC_REL where the order of the shared-memory atomics can change the rounding."""
    exact = _shared(tg, tl, T) <= 2
    same = (got.view(torch.int32) == ref.view(torch.int32)).all(2).all(0).cpu()
    rel = ((got.double() - ref.double()).norm(dim=(0, 2)) / ref.double().norm(dim=(0, 2)).clamp_min(1e-30)).cpu()
    print('%-58s %d sequences bit for bit (<= 2 terms per edge), %d within %.0e (max rel %.2e, %d of them bit for bit)'
          % (what, int(exact.sum()), int((~exact).sum()), ATOMIC_REL, rel[~exact].max().item() if (~exact).any() else 0.0,
             int(same[~exact].sum())))
    assert same[exact].all(), (what, torch.nonzero(exact & ~same).flatten().tolist())
    assert (rel[~exact] <= ATOMIC_REL).all(), (what, rel.max().item())


def _bits(a):
    return a.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ training distribution
@pytest.mark.parametrize('normalise', [True, False])
@pytest.mark.parametrize('n_base', [4, 5, 6])
def test_training_distribution(handles, n_base, normalise):
    T, N = 800, 8
    s = _scores(100 + n_base, T, N, n_base)
    tg, tl = _train_targets(10 + n_base, N, n_base)
    gl = torch.tensor([1.0, 0.0, -0.5, 1.0 / N, 2.0, 0.25, -1.0, 0.7])
    _compare('n_base %d, T %d, N %d' % (n_base, T, N), handles[n_base], n_base, s, tg, tl, gl, normalise)


def test_bench_shape_and_batch_position(handles):
    """N = 512, T = 800 with bench.py's targets: every sequence's loss and gradient against float64, and sequences 0, 255
    and 511 alone and in a permuted batch give the same loss bits and the same gradient (see _check_same: each of these
    targets has a state at 8 or more of its positions, so every sequence falls in the ATOMIC_REL case)."""
    n_base, T, N = 5, 800, 512
    h = handles[n_base]
    s = _scores(7, T, N, n_base)
    tg, tl = _train_targets(3, N, n_base)
    gl = torch.full((N,), 1.0 / N)
    loss = h.ctc_loss(s, tg, tl)
    grad = h.ctc_loss_bwd(s, tg, tl, gl)
    rl, rg = ts.ctc_loss_backward(s, tg, tl, gl, n_base)
    _check_loss('bench shape N 512: every sequence', loss, rl, NORM)
    _check('bench shape N 512: every sequence', grad, rg, gl, tl, NORM)
    del rl, rg
    for n in (0, 255, 511):
        one = slice(n, n + 1)
        l1 = h.ctc_loss(s[:, one], tg[one], tl[one])
        g1 = h.ctc_loss_bwd(s[:, one], tg[one], tl[one], gl[one])
        assert torch.equal(_bits(l1), _bits(loss[one])), n
        _check_same('bench shape: sequence %d alone' % n, g1, grad[:, one], tg[one], tl[one], T)
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(5))
    inv = perm.argsort()
    lp = h.ctc_loss(s[:, perm.cuda()], tg[perm], tl[perm])
    gp = h.ctc_loss_bwd(s[:, perm.cuda()], tg[perm], tl[perm], gl[perm])
    assert torch.equal(_bits(lp[inv.cuda()]), _bits(loss))
    _check_same('bench shape: permuted batch', gp[:, inv.cuda()], grad, tg, tl, T)


# ------------------------------------------------------------------------------------------------ block size and Lmax
# the backward raises NT = round_up(npos, 32) to ceil(S / 128) * 32 when 4 * NT < S: up to npos 64 for n_base 4 (S = 320),
# 160 for n_base 5 (S = 750) and 352 for n_base 6 (S = 1512).  Each alphabet's last raised npos and the next one.
_SWITCH = {4: (64, 65), 5: (160, 161), 6: (352, 353)}
_BLOCK_CASES = [(n, p) for n in (4, 5, 6) for p in sorted({1, 31, 32, 33, 383, 385, 1024} | set(_SWITCH[n]))]


@pytest.mark.parametrize('n_base,npos', _BLOCK_CASES)
def test_block_size_edges(handles, n_base, npos):
    """Lmax = npos + 2 at T = 1030, which makes the longest target (1023 moves) feasible.  One batch of full-width
    targets (len = Lmax and Lmax - 1) and one of short ones (len = Lmax // 4 and 3) with the same Lmax, each sequence
    held to the bounds of its own kind (see the module docstring)."""
    T, Lmax = MAX_T, npos + 2
    rs = np.random.RandomState(npos + 7 * n_base)
    h = handles[n_base]
    for kind, lens, gl in (('full width', [Lmax, max(3, Lmax - 1)], [1.0, -0.5]),
                           ('short', [max(3, Lmax // 4), 3], [0.25, 1.0])):
        tg, tl = _pad([rs.randint(1, n_base + 1, n) for n in lens], Lmax)
        s = _scores(npos + n_base + len(kind), T, 2, n_base)
        for normalise in (True, False):
            b = RAW if not normalise else NORM_LONG_SHORT if kind == 'short' or Lmax == 3 else NORM_LONG
            _compare('n_base %d, npos %d, %s' % (n_base, npos, kind), h, n_base, s, tg, tl, torch.tensor(gl), normalise,
                     b)


@pytest.mark.parametrize('n_base', [4, 5, 6])
def test_lmax_limit_refused(handles, n_base):
    """npos = Lmax - 2 must lie in 1..1024: Lmax = 1027 and Lmax = 2 raise XB_ERR_ARG from both directions, and nothing is
    launched (the backward used to launch the full-lattice posteriors and logZ before it checked Lmax)."""
    h = handles[n_base]
    T, N = 50, 2
    s = _scores(1, T, N, n_base)
    gl = torch.ones(N)
    for Lmax in (1027, 2):
        tg = torch.ones(N, Lmax, dtype=torch.int64)
        tl = torch.full((N,), min(Lmax, 40))
        for normalise in (True, False):
            before = h.launches
            with pytest.raises(RuntimeError, match=r'xb_ctc_crf_loss_fwd failed \(-1\)'):
                h.ctc_loss(s, tg, tl, normalise=normalise)
            with pytest.raises(RuntimeError, match=r'xb_ctc_crf_loss_bwd failed \(-1\)'):
                h.ctc_loss_bwd(s, tg, tl, gl, normalise=normalise)
            assert h.launches == before, (Lmax, normalise)


# ------------------------------------------------------------------------------------------------ time edges
@pytest.mark.parametrize('n_base', [4, 5, 6])
def test_time_edges(handles, n_base):
    """T = 1 and T = 2 with len 3, 4, 5 (T = 1, len 5 needs two moves in one step: no alignment), and T = 800 with a
    target of T + 3 bases: its one alignment moves at every step, so its log-sum is the sum of those move scores and its
    numerator is one edge per step."""
    h = handles[n_base]
    rs = np.random.RandomState(n_base)
    tg, tl = _pad([rs.randint(1, n_base + 1, n) for n in (3, 4, 5)], 5)
    gl = torch.tensor([1.0, -0.5, 0.25])
    for T in (1, 2):
        s = _scores(T + n_base, T, 3, n_base)
        for normalise in (True, False):
            loss, _ = _compare('n_base %d, T %d, len 3..5' % (n_base, T), h, n_base, s, tg, tl, gl, normalise)
            if T == 1:
                assert loss[2].item() == np.float32(1e38) / np.float32(5)
    T = 800
    one = rs.randint(1, n_base + 1, T + 3)
    tg, tl = _pad([one, rs.randint(1, n_base + 1, 400)], T + 3)
    gl = torch.tensor([1.0, 0.5])
    s = _scores(33 + n_base, T, 2, n_base)
    for normalise in (True, False):
        loss, grad = _compare('n_base %d, T 800, len T + 3' % n_base, h, n_base, s, tg, tl, gl, normalise)
        r = [max(v - 1, 0) for v in one]
        state = [(r[j] * n_base + r[j + 1]) * n_base + r[j + 2] for j in range(T + 1)]
        edge = torch.tensor([state[t + 1] * (n_base + 1) + r[t] + 1 for t in range(T)], device='cuda')
        s64 = s[:, 0].double()
        path = s64.gather(1, edge[:, None])[:, 0]
        num = torch.zeros_like(s64).scatter_(1, edge[:, None], 1.0)
        den = torch.zeros_like(s64)
        if normalise:
            path = path - bo.CRF(3, ALPHABETS[n_base]).logZ(s[:, :1].double().cpu()).item() / T
            den = h.posteriors(s)[:, 0].double()
        b = NORM if normalise else RAW
        _check_loss('n_base %d, T 800, len T + 3: sum of move scores' % n_base, loss[:1], -path.sum()[None] / (T + 3), b)
        _check('n_base %d, T 800, len T + 3: one-hot numerator' % n_base, grad[:, :1], ((den - num) / (T + 3))[:, None],
               gl[:1], tl[:1], b)


# ------------------------------------------------------------------------------------------------ collisions, padding
@pytest.mark.parametrize('n_base', [4, 5, 6])
def test_colliding_edges(handles, n_base):
    """Homopolymers and 2-base repeats of 400 bases at T = 800: every position shares its stay and its move edge with
    hundreds of others, so each step adds many numerator terms to one edge of the shared row."""
    T, L = 800, 400
    x = 5 if n_base >= 5 else 4                                # X where the alphabet has it
    tg, tl = _pad([[1] * L, [x] * L, [1, 2] * (L // 2), [x, 1] * (L // 2)], L)
    gl = torch.tensor([1.0, 0.5, -1.0, 0.25])
    s = _scores(55 + n_base, T, 4, n_base)
    for normalise in (True, False):
        _compare('n_base %d, homopolymers and repeats' % n_base, handles[n_base], n_base, s, tg, tl, gl, normalise)


def test_padding_and_garbage(handles):
    """The same targets at their exact width, padded to Lmax + 200 with zeros, and with garbage labels (1..n_base and
    negative values, which clamp to 0 as padding does) after each length: same loss bits, same gradient.  Row 0 is a
    de Bruijn target, in which no two positions share an edge: its gradient is the same bit for bit."""
    n_base, T, N = 5, 800, 6
    h = handles[n_base]
    tg, tl = _train_targets(21, N - 1, n_base)
    rows = [_de_bruijn(n_base)] + [r[:n].tolist() for r, n in zip(tg, tl)]
    width = max(len(r) for r in rows)
    exact, tl = _pad(rows, width)
    padded, _ = _pad(rows, width + 200)
    rs = np.random.RandomState(4)
    garbage = torch.from_numpy(rs.choice([-3, -1] + list(range(1, n_base + 1)), size=(N, width + 200)))
    for i, n in enumerate(tl.tolist()):
        garbage[i, :n] = exact[i, :n]
    s = _scores(61, T, N, n_base)
    gl = torch.tensor([1.0, 0.5, -1.0, 0.25, 1.0 / N, 2.0])
    for normalise in (True, False):
        loss, grad = _compare('padding: exact width', h, n_base, s, exact, tl, gl, normalise)
        for name, tgt in (('zeros', padded), ('garbage', garbage)):
            l2 = h.ctc_loss(s, tgt, tl, normalise=normalise)
            g2 = h.ctc_loss_bwd(s, tgt, tl, gl, normalise=normalise)
            assert torch.equal(_bits(l2), _bits(loss)), name
            _check_same('padded with %s, normalise=%d' % (name, normalise), g2, grad, exact, tl, T)
        assert _shared(exact[:1], tl[:1], T).item() == 1


# ------------------------------------------------------------------------------------------------ infeasible targets
@pytest.mark.parametrize('normalise', [True, False])
def test_infeasible_and_degenerate_lengths(handles, normalise):
    """len = T + 4 (more moves than steps) and len = 1, 2 (< state_len) among feasible sequences.  The kernels' contract
    (seqdist's semiring zero, -1e38): loss = 1e38 / len in fp32, and a gradient without a numerator, that is
    grad_loss / len * P_den with normalise and exactly zero without.  Through CTC_CRF.ctc_loss with loss_clip such a
    sequence's gradient is exactly zero, and the batch's other sequences are those of a batch without them."""
    from xna_basecaller_b200.crf.model import CTC_CRF
    n_base, T = 5, 400
    h = handles[n_base]
    tg, tl = _train_targets(8, 4, n_base, 150, 250)
    rs = np.random.RandomState(9)
    bad = [rs.randint(1, n_base + 1, T + 4).tolist(), [2], [3, 1]]
    rows = [tg[0, :tl[0]].tolist(), bad[0], tg[1, :tl[1]].tolist(), bad[1], tg[2, :tl[2]].tolist(), bad[2],
            tg[3, :tl[3]].tolist()]
    tg, tl = _pad(rows, T + 4)
    inf, ok = [1, 3, 5], [0, 2, 4, 6]
    gl = torch.tensor([1.0, 0.5, -0.5, 2.0, 0.25, -1.0, 1.0 / 7])
    s = _scores(70, T, len(rows), n_base)
    loss, grad = _compare('infeasible lengths', h, n_base, s, tg, tl, gl, normalise)
    want = torch.full((3,), 1e38, dtype=torch.float32) / tl[inf].float()
    assert torch.equal(_bits(loss[inf].cpu()), _bits(want))
    assert torch.isfinite(grad).all()
    if normalise:
        post = h.posteriors(s)
        for n in inf:
            assert torch.equal(_bits(grad[:, n]), _bits(post[:, n] * (gl[n] / tl[n].float()).item()))
    else:
        assert not grad[:, inf].any()
    l2 = h.ctc_loss(s[:, ok], tg[ok], tl[ok], normalise=normalise)
    g2 = h.ctc_loss_bwd(s[:, ok], tg[ok], tl[ok], gl[ok], normalise=normalise)
    assert torch.equal(_bits(l2), _bits(loss[ok]))
    _check_same('infeasible lengths: the others alone, normalise=%d' % normalise, g2, grad[:, ok], tg[ok], tl[ok], T)
    crf = CTC_CRF(3, ALPHABETS[n_base])
    sr = s.clone().requires_grad_()
    out = crf.ctc_loss(sr, tg.cuda(), tl.cuda(), loss_clip=100.0, reduction='none', normalise_scores=normalise)
    out.backward(gl.cuda())
    clipped = ((loss < 0) | (loss > 100.0)).cpu()
    assert clipped[inf].all()
    for n in range(len(rows)):
        assert bool(sr.grad[:, n].any()) != bool(clipped[n]), n
    crf.engine.close()


# ------------------------------------------------------------------------------------------------ plugin route
def test_plugin_route(handles):
    """CTC_CRF.ctc_loss with reduction 'mean' (grad_loss 1/N) and 'none' (any grad_loss), on fp32 scores and on fp16
    scores (whose gradient _CTCLoss.backward casts to fp16): the gradient is Handle.ctc_loss_bwd's, bit for bit or within
    ATOMIC_REL as _check_same decides -- after the fp16 cast, within one fp16 rounding step where it is not bit for bit;
    and loss_clip zeroes exactly the gradients of the sequences whose loss it clips."""
    from xna_basecaller_b200.crf.model import CTC_CRF
    n_base, T, N = 5, 800, 8
    h = handles[n_base]
    crf = CTC_CRF(3, ALPHABETS[n_base])
    tg, tl = _train_targets(30, N - 1, n_base)
    rows = [_de_bruijn(n_base)] + [r[:n].tolist() for r, n in zip(tg, tl)]
    tg, tl = _pad(rows, max(len(r) for r in rows))
    exact = (_shared(tg, tl, T) <= 2).cuda()
    s = _scores(80, T, N, n_base)
    w = torch.tensor([1.0, -0.5, 0.25, 2.0, 0.0, 1.0, -1.0, 0.3])
    for dtype in (torch.float32, torch.float16):
        sx = s.to(dtype)
        for reduction in ('mean', 'none'):
            sr = sx.clone().requires_grad_()
            out = crf.ctc_loss(sr, tg.cuda(), tl.cuda(), reduction=reduction)
            gl = torch.full((N,), 1.0 / N) if reduction == 'mean' else w
            out.backward() if reduction == 'mean' else out.backward(gl.cuda())
            assert sr.grad.dtype == dtype
            direct = h.ctc_loss_bwd(sx.float(), tg, tl, gl)
            what = 'plugin %s, %s' % (reduction, str(dtype)[6:])
            if dtype == torch.float32:
                _check_same(what, sr.grad, direct, tg, tl, T)
                continue
            got = sr.grad.float()
            assert torch.equal(got[:, exact], direct[:, exact].half().float()), what
            ulp = torch.ldexp(torch.ones_like(direct), (torch.frexp(direct)[1] - 11).clamp_min(-24))
            diff = (got - direct).abs()
            print('%-58s max |fp16 - fp32| / fp16 ulp %.2f where not bit for bit' % (what, (diff / ulp)[:, ~exact].max()))
            assert (diff <= ulp).all(), what
    loss = h.ctc_loss(s, tg, tl)
    clip = float(loss.median())
    sr = s.clone().requires_grad_()
    out = crf.ctc_loss(sr, tg.cuda(), tl.cuda(), loss_clip=clip, reduction='none')
    assert torch.equal(_bits(out.detach()), _bits(loss.clamp(0.0, clip)))
    out.backward(w.cuda())
    clipped = ((loss < 0) | (loss > clip) | (w.cuda() == 0)).cpu()
    assert 0 < int(clipped.sum()) < N
    for n in range(N):
        assert bool(sr.grad[:, n].any()) != bool(clipped[n]), n
    crf.engine.close()
