"""CPU restatement (torch fp32/fp64 + numpy) of ub-bonito's basecalling forward path.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Every function cites the reference lines it
follows (paths relative to /root/reference/ub-bonito/).  The restatement is written to be read
next to the reference, not copied from it: tensors are handled functionally from a plain
``state_dict`` instead of through nn.Module classes, and the CRF recursions are explicit
alpha/beta loops instead of seqdist's autograd formulation (``oracle.seqdist_restated`` keeps
the autograd form; tests check the two against each other and against brute force).
"""
from itertools import groupby

import numpy as np
import torch
import torch.nn.functional as F

NEG = -1e38   # seqdist semiring "zero" (core.Log.zero / core.Max.zero)


# ----------------------------------------------------------------------------- encoder
def swish(x):
    """bonito/nn.py:23-25 (Swish = torch.nn.SiLU)."""
    return x * torch.sigmoid(x)


def conv_stem(sd, x):
    """Three Convolution layers, bonito/nn.py:57-68 built at bonito/crf/model.py:138-139,148-150:
    (1->4,k5,p2), (4->16,k5,p2), (16->features,k19,s5,p9), each followed by swish.
    x: (N, 1, L) -> (N, features, L//5)."""
    y = swish(F.conv1d(x, sd['encoder.0.conv.weight'], sd['encoder.0.conv.bias'], padding=2))
    y = swish(F.conv1d(y, sd['encoder.1.conv.weight'], sd['encoder.1.conv.bias'], padding=2))
    w = sd['encoder.2.conv.weight']
    y = swish(F.conv1d(y, w, sd['encoder.2.conv.bias'], stride=5, padding=w.shape[-1] // 2))
    return y


def lstm_layer(x, w_ih, w_hh, b_ih, b_hh, reverse):
    """One bonito LSTM layer: bonito/nn.py:176-235, forward at :189-193.
    Single-layer unidirectional torch.nn.LSTM, gate order i,f,g,o, zero initial state; a
    reversed layer walks time from T-1 down to 0 (the reference flips input and output).
    x: (T, N, F) -> (T, N, H)."""
    T, N, _ = x.shape
    H = w_hh.shape[1]
    gin = x @ w_ih.t() + (b_ih + b_hh)
    h = x.new_zeros(N, H)
    c = x.new_zeros(N, H)
    out = x.new_empty(T, N, H)
    order = range(T - 1, -1, -1) if reverse else range(T)
    for t in order:
        g = gin[t] + h @ w_hh.t()
        i, f, gg, o = g.split(H, dim=1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
        h = torch.sigmoid(o) * torch.tanh(c)
        out[t] = h
    return out


def lstm_layer_library(x, w_ih, w_hh, b_ih, b_hh, reverse):
    """Same layer through torch's own LSTM op (what the reference actually executes on CPU);
    used for the timed CPU baseline."""
    N = x.shape[1]
    H = w_hh.shape[1]
    if reverse:
        x = x.flip(0)
    hx = (x.new_zeros(1, N, H), x.new_zeros(1, N, H))
    y, _, _ = torch._VF.lstm(x, hx, [w_ih, w_hh, b_ih, b_hh], True, 1, 0.0, False, False, False)
    if reverse:
        y = y.flip(0)
    return y


LSTM_DIRECTIONS = (True, False, True, False, True)   # bonito/crf/model.py:152-154


def lstm_stack(sd, x, library=False):
    """encoder.4 .. encoder.8: reverse, forward, reverse, forward, reverse."""
    fn = lstm_layer_library if library else lstm_layer
    for layer, rev in zip(range(4, 9), LSTM_DIRECTIONS):
        p = 'encoder.%d.rnn.' % layer
        x = fn(x, sd[p + 'weight_ih_l0'], sd[p + 'weight_hh_l0'], sd[p + 'bias_ih_l0'],
               sd[p + 'bias_hh_l0'], rev)
    return x


def crf_head(sd, x, n_base, scale=5.0, blank_score=2.0, expand_blanks=True):
    """LinearCRFEncoder.forward, bonito/nn.py:112-133 (no extra_linear, dropout off):
    scale*tanh(x W^T + b), then a constant blank score inserted as entry 0 of every group of
    n_base (so each state gets n_base+1 incoming-edge scores)."""
    s = torch.tanh(x @ sd['encoder.9.linear.weight'].t() + sd['encoder.9.linear.bias']) * scale
    if blank_score is not None and expand_blanks:
        T, N, C = s.shape
        s = s.reshape(T, N, C // n_base, n_base)
        blank = s.new_full((T, N, C // n_base, 1), blank_score)
        s = torch.cat([blank, s], dim=-1).reshape(T, N, -1)
    return s


def encoder_forward(sd, x, n_base, scale=5.0, blank_score=2.0, library=False):
    """Model.forward, bonito/crf/model.py:212-213: (N,1,L) -> (T, N, C*NZ)."""
    y = conv_stem(sd, x).permute(2, 0, 1)          # Permute([2,0,1]), bonito/nn.py:156-167
    y = lstm_stack(sd, y.contiguous(), library=library)
    return crf_head(sd, y, n_base, scale, blank_score)


def reference_state_dict(n_base=5, state_len=3, features=768, seed=0, head_gain=12.0, head_shift=-3.0,
                         wih_gain=2.0, whh_gain=0.4, dtype=torch.float32):
    """Deterministic random weights with the reference's state_dict keys and shapes
    (SURVEY.md section 5 checkpoint row).  Plain seeded normals (no QR / LAPACK), so the same
    weights are regenerated bit-identically on any machine with the same torch build.
    The default gains are chosen so that the decoded strings depend on the input signal and mix
    blanks with moves (the reference's own orthogonal init decodes to the empty string, and
    unit-gain recurrences fall into an input-independent limit cycle)."""
    g = torch.Generator().manual_seed(seed)

    def rnd(*shape, std):
        return (torch.randn(*shape, generator=g, dtype=torch.float32) * std).to(dtype)

    sd = {}
    sd['encoder.0.conv.weight'] = rnd(4, 1, 5, std=0.45)
    sd['encoder.0.conv.bias'] = rnd(4, std=0.3)
    sd['encoder.1.conv.weight'] = rnd(16, 4, 5, std=0.22)
    sd['encoder.1.conv.bias'] = rnd(16, std=0.2)
    sd['encoder.2.conv.weight'] = rnd(features, 16, 19, std=0.057)
    sd['encoder.2.conv.bias'] = rnd(features, std=0.05)
    for layer in range(4, 9):
        p = 'encoder.%d.rnn.' % layer
        sd[p + 'weight_ih_l0'] = rnd(4 * features, features, std=wih_gain * features ** -0.5)
        sd[p + 'weight_hh_l0'] = rnd(4 * features, features, std=whh_gain * features ** -0.5)
        sd[p + 'bias_ih_l0'] = rnd(4 * features, std=0.5).clamp_(-1, 1)
        sd[p + 'bias_hh_l0'] = torch.zeros(4 * features, dtype=dtype)   # bonito/nn.py:209-213
    size = n_base ** (state_len + 1)
    sd['encoder.9.linear.weight'] = rnd(size, features, std=head_gain * features ** -0.5)
    sd['encoder.9.linear.bias'] = rnd(size, std=0.02 * head_gain) + head_shift
    return sd


# ----------------------------------------------------------------------------- CTC-CRF
def crf_idx(n_base, state_len):
    """CTC_CRF.idx, bonito/crf/model.py:31-36.  Row c lists the source state of each of the
    NZ = n_base+1 edges entering state c: k=0 is the stay/blank edge (source c); k=1+j is a move
    that dropped leading base j: source = j * n_base^(state_len-1) + c // n_base."""
    C = n_base ** state_len
    c = np.arange(C)
    moves = np.arange(n_base)[None, :] * n_base ** (state_len - 1) + (c // n_base)[:, None]
    return torch.from_numpy(np.concatenate([c[:, None], moves], axis=1).astype(np.int32))


class CRF:
    """CTC_CRF, bonito/crf/model.py:24-135, over explicit alpha/beta recursions."""

    def __init__(self, state_len, alphabet):
        self.alphabet = list(alphabet)
        self.state_len = state_len
        self.n_base = len(alphabet) - 1
        self.NZ = self.n_base + 1
        self.C = self.n_base ** state_len
        self.idx = crf_idx(self.n_base, state_len).to(torch.int64)
        flat = self.idx.flatten().argsort(stable=True)
        self.src_edges = flat.reshape(self.C, self.NZ)       # edges leaving each state
        self.src_dst = self.src_edges // self.NZ             # and the states they enter

    # -- scans (seqdist.sparse semantics, see oracle/seqdist_restated.py) ---------------
    @staticmethod
    def _sum(x, semiring):
        return torch.logsumexp(x, dim=-1) if semiring == 'log' else x.max(dim=-1)[0]

    def _Ms(self, scores):
        T, N, _ = scores.shape
        return scores.reshape(T, N, self.C, self.NZ)          # crf/model.py:43

    def forward_scores(self, scores, semiring='log'):
        """crf/model.py:51-55; alpha_0 = one (0) for every state (:44)."""
        Ms = self._Ms(scores)
        T, N = Ms.shape[:2]
        alpha = Ms.new_zeros(T + 1, N, self.C)
        for t in range(T):
            alpha[t + 1] = self._sum(Ms[t] + alpha[t][:, self.idx], semiring)
        return alpha

    def backward_scores(self, scores, semiring='log'):
        """crf/model.py:57-61; beta_T = one (0) for every state (:45)."""
        T, N, _ = scores.shape
        beta = scores.new_zeros(T + 1, N, self.C)
        for t in range(T - 1, -1, -1):
            beta[t] = self._sum(scores[t][:, self.src_edges] + beta[t + 1][:, self.src_dst], semiring)
        return beta

    def logZ(self, scores, semiring='log'):
        """crf/model.py:41-46: sum over final states of alpha_T (+ beta_T = 0)."""
        return self._sum(self.forward_scores(scores, semiring)[-1], semiring)

    def edge_marginals(self, scores, semiring='log'):
        """(Ms + alpha_t[idx]) + beta_{t+1}: the quantity seqdist applies dsum to (T,N,C,NZ)."""
        Ms = self._Ms(scores)
        a = self.forward_scores(scores, semiring)
        b = self.backward_scores(scores, semiring)
        return (Ms + a[:-1][:, :, self.idx]) + b[1:, :, :, None]

    def posteriors(self, scores, semiring='log'):
        """SequenceDist.posteriors = d(sum_n logZ)/d scores (crf/model.py:93,216): softmax over all
        C*NZ edges of a step for Log, one-hot at the first arg-max for Max."""
        T, N, _ = scores.shape
        x = self.edge_marginals(scores, semiring).reshape(T, N, -1)
        if semiring == 'log':
            return torch.softmax(x, dim=2)
        return torch.zeros_like(x).scatter_(2, x.argmax(2, keepdim=True), 1.0)

    def viterbi(self, scores):
        """crf/model.py:92-95: arg-max edge of the max-marginals, reported as edge % NZ: 0 = blank,
        j+1 = a move whose DROPPED base is j."""
        T, N, _ = scores.shape
        x = self.edge_marginals(scores, 'max').reshape(T, N, -1)
        return x.argmax(2) % self.NZ

    def path_to_str(self, path):
        """crf/model.py:97-100: every non-zero label emits one letter, no repeat collapsing."""
        letters = np.frombuffer(''.join(self.alphabet).encode(), dtype='u1')
        path = np.asarray(path)
        return letters[path[path != 0]].tobytes().decode()

    def decode_batch(self, scores):
        """SeqdistModel.decode_batch, crf/model.py:215-218."""
        post = self.posteriors(scores.to(torch.float32), 'log') + 1e-8
        paths = self.viterbi(post.log()).to(torch.int16).T
        return [self.path_to_str(p) for p in paths.numpy()]

    # -- training loss ------------------------------------------------------------------
    def normalise(self, scores):
        """crf/model.py:48-49."""
        return scores - self.logZ(scores)[:, None] / len(scores)

    def prepare_ctc_scores(self, scores, targets, dtype=torch.float32):
        """crf/model.py:102-116.  targets are 1-based labels, 0-padded.  The reference casts to float32; the float64
        references pass dtype=torch.float64."""
        tg = torch.clamp(targets - 1, 0)
        T = scores.shape[0]
        scores = scores.to(dtype)
        n = tg.size(1) - (self.state_len - 1)
        state = torch.zeros_like(tg[:, :n])
        for i in range(self.state_len):
            state = state * self.n_base + tg[:, i:n + i]
        stay_idx = state * self.NZ
        move_idx = stay_idx[:, 1:] + tg[:, :n - 1] + 1
        stay = scores.gather(2, stay_idx.expand(T, -1, -1))
        move = scores.gather(2, move_idx.expand(T, -1, -1))
        return stay, move

    @staticmethod
    def simple_logZ(stay, move, lengths):
        """seqdist.ctc_simple.logZ_cupy (crf/model.py:122): log-sum over monotone alignments that
        start at position 0 and sit at position lengths-1 after the last step."""
        T, N, L = stay.shape
        a = stay.new_full((N, L), NEG)
        a[:, 0] = 0.0
        for t in range(T):
            moved = torch.cat([a.new_full((N, 1), NEG), move[t] + a[:, :-1]], dim=1)
            a = torch.logsumexp(torch.stack([stay[t] + a, moved], dim=-1), dim=-1)
        return a[torch.arange(N), lengths.to(torch.int64) - 1]

    def ctc_loss(self, scores, targets, target_lengths, loss_clip=None, reduction='mean',
                 normalise_scores=True):
        """crf/model.py:118-131."""
        if normalise_scores:
            scores = self.normalise(scores)
        stay, move = self.prepare_ctc_scores(scores, targets)
        logz = self.simple_logZ(stay, move, target_lengths + 1 - self.state_len)
        loss = -(logz / target_lengths)
        if loss_clip:
            loss = torch.clamp(loss, 0.0, loss_clip)
        if reduction == 'mean':
            return loss.mean()
        if reduction in ('none', None):
            return loss
        raise ValueError('Unknown reduction type {}'.format(reduction))

    # -- rarely used surface (SURVEY 8a-14, a-15) ----------------------------------------
    def reverse_complement(self, scores):
        """crf/model.py:78-90."""
        T, N, _ = scores.shape
        n, sl = self.n_base, self.state_len
        s = scores.reshape(T, N, *([n] * sl), n + 1)
        blanks = s[..., 0].permute(0, 1, *range(sl + 1, 1, -1)).reshape(T, N, -1, 1).flip([0, 2])
        emis = s[..., 1:].permute(0, 1, *range(sl, 1, -1), sl + 2, sl + 1).reshape(T, N, -1, n)
        emis = emis.flip([0, 2, 3])
        return torch.cat([blanks, emis], dim=-1).reshape(T, N, -1)

    def compute_transition_probs(self, scores, betas):
        """crf/model.py:63-76."""
        T, N, _ = scores.shape
        lt = self._Ms(scores) + betas[1:, :, :, None]
        lt = torch.cat([lt[:, :, :, [0]],
                        lt[:, :, :, 1:].transpose(3, 2).reshape(T, N, -1, self.n_base)], dim=-1)
        return torch.softmax(lt, dim=-1), torch.softmax(betas[0], dim=-1)


# ----------------------------------------------------------------------------- chunking / stitching
def chunk(signal, chunksize, overlap):
    """bonito/util.py:152-166.  signal: 1-D tensor -> (n_chunks, 1, chunksize)."""
    T = signal.shape[0]
    if chunksize == 0:
        out = signal[None, :]
    elif T < chunksize:
        out = torch.cat([signal.new_zeros(chunksize - T), signal])[None, :]     # left pad (:160)
    else:
        step = chunksize - overlap
        stub = (T - overlap) % step
        starts = list(range(stub, T - chunksize + 1, step))
        out = torch.stack([signal[s:s + chunksize] for s in starts])
        if stub > 0:
            out = torch.cat([signal[None, :chunksize], out], dim=0)             # leading stub chunk
    return out.unsqueeze(1)


def stitch_plan(n_chunks, chunksize, overlap, length, stride):
    """Slices (lo, hi) per chunk that bonito/util.py:169-188 concatenates (forward direction)."""
    if n_chunks == 1:
        return [(0, None)]
    semi = overlap // 2
    start, end = semi // stride, (chunksize - semi) // stride
    stub = (length - overlap) % (chunksize - overlap)
    first_end = (stub + semi) // stride if stub > 0 else end
    return [(0, first_end)] + [(start, end)] * (n_chunks - 2) + [(start, None)]


def stitch(chunks, chunksize, overlap, length, stride, reverse=False):
    """bonito/util.py:169-188 for array-like chunks (n_chunks, T)."""
    if chunks.shape[0] == 1:
        return chunks[0]
    cat = np.concatenate if isinstance(chunks, np.ndarray) else torch.cat
    if reverse:
        semi = overlap // 2
        start, end = semi // stride, (chunksize - semi) // stride
        stub = (length - overlap) % (chunksize - overlap)
        first_end = (stub + semi) // stride if stub > 0 else end
        parts = [chunks[-1][:-start]] + [x[-end:-start] for x in reversed(list(chunks[1:-1]))]
        parts.append(chunks[0][-first_end:])
        return cat(parts)
    plan = stitch_plan(chunks.shape[0], chunksize, overlap, length, stride)
    return cat([chunks[i][lo:hi] for i, (lo, hi) in enumerate(plan)])


def batchify(items, batchsize):
    """bonito/util.py:191-210 for (key, tensor-of-chunks) items: exact-size batches, each with the
    list of (key, (row_start, row_end)) spans it holds."""
    held, fill = [], 0
    for key, v in items:
        off = 0
        while off < len(v):
            take = min(batchsize - fill, len(v) - off)
            held.append(((key, (fill, fill + take)), v[off:off + take]))
            fill += take
            off += take
            if fill == batchsize:
                yield tuple(k for k, _ in held), torch.cat([x for _, x in held])
                held, fill = [], 0
    if held:
        yield tuple(k for k, _ in held), torch.cat([x for _, x in held])


def unbatchify(batches):
    """bonito/util.py:213-225: regroup consecutive spans with the same key (values are dicts of
    arrays indexed by batch row)."""
    def spans():
        for keys, v in batches:
            for key, (lo, hi) in keys:
                yield key, {name: arr[lo:hi] for name, arr in v.items()}
    for key, grp in groupby(spans(), key=lambda kv: kv[0]):
        parts = [p for _, p in grp]
        merged = {}
        for name in parts[0]:
            vals = [p[name] for p in parts]
            merged[name] = np.concatenate(vals) if isinstance(vals[0], np.ndarray) else torch.cat(vals)
        yield key, merged


def left_pack(strings, T):
    """bonito/crf/basecall.py:56-82 (Viterbi branch): ord() of each decoded string left-packed
    into (N, T) int8, qstring 'O' at the same positions, all-False moves."""
    N = len(strings)
    seq = np.zeros((N, T), dtype=np.int8)
    qs = np.zeros((N, T), dtype=np.int8)
    for i, s in enumerate(strings):
        seq[i, :len(s)] = np.frombuffer(s.encode(), dtype='u1')
        qs[i, :len(s)] = ord('O')
    return {'sequence': seq, 'qstring': qs, 'moves': np.zeros((N, T), dtype=bool)}


def to_str(x):
    """koi.decode.to_str as used at bonito/crf/basecall.py:90-91: drop zeros, bytes -> ascii."""
    x = np.asarray(x)
    return x[x != 0].astype('u1').tobytes().decode('ascii')


def basecall(score_fn, crf, reads, chunksize, overlap, batchsize, stride=5):
    """bonito/crf/basecall.py:96-119 run synchronously.  reads: iterable of (read_id, 1-D float32
    numpy signal); score_fn(batch (N,1,cs) tensor) -> (T,N,C*NZ) scores.  Yields
    (read_id, {'sequence','qstring','sig_move'})."""
    def chunks():
        for rid, sig in reads:
            yield (rid, len(sig)), chunk(torch.from_numpy(sig), chunksize, overlap)

    def scored():
        for keys, batch in batchify(chunks(), batchsize):
            scores = score_fn(batch)
            yield keys, left_pack(crf.decode_batch(scores), scores.shape[0])

    for (rid, length), attrs in unbatchify(scored()):
        st = {k: stitch(v, chunksize, overlap, length, stride) for k, v in attrs.items()}
        moves = np.asarray(st['moves'], dtype=bool)
        sig_move = np.full(moves.size * stride, False)
        sig_move[np.where(moves)[0] * stride] = True
        yield rid, {'sequence': to_str(st['sequence']), 'qstring': to_str(st['qstring']),
                    'sig_move': sig_move}
