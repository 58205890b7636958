"""float64 references of the training gradient one part at a time: the CTC-CRF loss and its gradient w.r.t. the scores
(xb_ctc_crf_loss_fwd / _bwd), and the three stages of the encoder backward (xb_encoder_bwd_stages): the CRF head, one
LSTM layer and the convolution stem.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Every function is plain torch and runs on whatever device its inputs live on: the GPU tests run them there, because a
T = 800 LSTM layer in float64 on the CPU takes minutes.  Inputs are the stage's exact 16-bit inputs as float64 and the
weights the handle holds (`held`): fp16-rounded, or bf16-rounded for a handle created with bf16=True.

`lstm_backward_matched` is the LSTM layer's backward written out step by step, with the roundings of csrc/lstm_bptt.cu and
csrc/train_bwd.cu at the places the kernels round; with rounded=False it is the exact float64 backward (the CPU tests pin
that against autograd).
"""
import torch

from oracle import bonito_oracle as bo

F64 = torch.float64


def held(w, bf16=False):
    """The value of an fp32 weight as the handle's forward kernels multiply it, as float64."""
    w = w.float()
    if bf16:
        w = w.bfloat16().float()
    return w.half().to(F64)


def held_bwd(w):
    """The value of an fp32 weight in the handle's transposed backward copies (bf16 rounded from the fp32 weight)."""
    return w.float().bfloat16().to(F64)


def _grads(out, cot, inputs):
    gs = torch.autograd.grad(out, inputs, cot, allow_unused=True)
    return [torch.zeros_like(i) if g is None else g for i, g in zip(inputs, gs)]


# ----------------------------------------------------------------------------------------------------------- CTC-CRF loss
def ctc_loss_backward(scores, targets, lengths, grad_loss, n_base, normalise=True, state_len=3):
    """CTC_CRF.ctc_loss(reduction='none') (bonito/crf/model.py:102-131) and its gradient, in float64.

    scores (T, N, S = n_base^state_len * (n_base + 1)), targets (N, Lmax) 1-based labels, lengths (N,), grad_loss (N,)
    -> (loss (N,), dscores (T, N, S)): loss[n] = -logZ_n / lengths[n], logZ_n the log-sum over the alignments of target n
    (of the scores less logZ / T with normalise), and dscores = d(sum_n grad_loss[n] * loss[n]) / d scores in the closed
    form (P_den - P_num) * grad_loss / length: P_den the edge posteriors of the full lattice (only with normalise), P_num
    those of the target's alignment lattice, from explicit alpha / beta recursions over the target positions.

    A target no alignment reaches follows the kernels' contract, which is seqdist's semiring zero (-1e38): its loss is
    1e38 / length and it has no P_num term.  That is the case for length < state_len (no end position), length > Lmax,
    and more moves than steps (length - state_len > T).  Autograd through the reference would instead spread a numerator
    over paths of score ~-1e38, and index the end position with a negative number when length < state_len."""
    dev = scores.device
    T, N, S = scores.shape
    NZ = n_base + 1
    crf = bo.CRF(state_len, range(NZ))
    crf.idx, crf.src_edges, crf.src_dst = (t.to(dev) for t in (crf.idx, crf.src_edges, crf.src_dst))
    s = scores.to(F64)
    p_den = None
    if normalise:
        p_den = crf.posteriors(s)
        s = crf.normalise(s)
    # the alignment lattice (crf/model.py:102-116): stay edge of every position and the move edge into positions 1..
    tg = targets.to(dev, torch.int64).clamp_min(1) - 1
    npos = tg.shape[1] - (state_len - 1)
    state = torch.zeros_like(tg[:, :npos])
    for i in range(state_len):
        state = state * n_base + tg[:, i:npos + i]
    stay_idx = state * NZ
    move_idx = stay_idx[:, 1:] + tg[:, :npos - 1] + 1
    stay = s.gather(2, stay_idx.expand(T, -1, -1))
    move = s.gather(2, move_idx.expand(T, -1, -1))
    alpha = s.new_full((T + 1, N, npos), bo.NEG)
    alpha[0, :, 0] = 0.0
    for t in range(T):
        a = stay[t] + alpha[t]
        a[:, 1:] = torch.logaddexp(a[:, 1:], move[t] + alpha[t, :, :-1])
        alpha[t + 1] = a
    length = lengths.to(dev, torch.int64)
    last = length - state_len
    reach = (last >= 0) & (last < npos)
    end = last.clamp(0, npos - 1)
    z = torch.where(reach, alpha[T, torch.arange(N, device=dev), end], torch.full_like(alpha[T, :, 0], bo.NEG))
    feasible = reach & (z > -1e37)
    loss = -z / length
    beta = s.new_full((T + 1, N, npos), bo.NEG)
    beta[T, torch.arange(N, device=dev)[feasible], end[feasible]] = 0.0
    for t in range(T - 1, -1, -1):
        b = stay[t] + beta[t + 1]
        b[:, :-1] = torch.logaddexp(b[:, :-1], move[t] + beta[t + 1, :, 1:])
        beta[t] = b
    zf = torch.where(feasible, z, 0.0)[:, None]
    keep = feasible[:, None]
    p_stay = torch.where(keep, torch.exp(alpha[:-1] + stay + beta[1:] - zf), 0.0)
    p_move = torch.where(keep, torch.exp(alpha[:-1, :, :-1] + move + beta[1:, :, 1:] - zf), 0.0)
    p_num = s.new_zeros(T, N, S)
    p_num.scatter_add_(2, stay_idx.expand(T, -1, -1), p_stay)
    p_num.scatter_add_(2, move_idx.expand(T, -1, -1), p_move)
    d = -p_num if p_den is None else p_den - p_num
    return loss, d * (grad_loss.to(dev, F64) / length)[:, None]


# ----------------------------------------------------------------------------------------------------------- CRF head
def crf_head_backward(x, w, b, dscores, n_base, scale=5.0, blank_score=2.0):
    """LinearCRFEncoder (bonito/nn.py:112-133) through scale * tanh and the blank expansion.
    x (T, N, 768), w (n_base^4, 768), b (n_base^4,), dscores (T, N, C * NZ) -> (dw, db, dx), float64."""
    x, w, b = (t.to(F64).detach().requires_grad_() for t in (x, w, b))
    s = bo.crf_head({'encoder.9.linear.weight': w, 'encoder.9.linear.bias': b}, x, n_base, scale, blank_score)
    dw, db, dx = _grads(s, dscores.to(F64), [w, b, x])
    return dw, db, dx


# ----------------------------------------------------------------------------------------------------------- conv stem
def conv_stem_backward(signal, w1, b1, w2, b2, w3, b3, dy):
    """Three convolutions with swish, then Permute([2, 0, 1]) (bonito/nn.py:57-68, 156-167).
    signal (N, L); dy (T, N, 768) the gradient w.r.t. the stem output -> [dw1, db1, dw2, db2, dw3 (768, 16, 19), db3]."""
    ps = [t.to(F64).detach().requires_grad_() for t in (w1, b1, w2, b2, w3, b3)]
    keys = ['encoder.%d.conv.%s' % (i, k) for i in range(3) for k in ('weight', 'bias')]
    y = bo.conv_stem(dict(zip(keys, ps)), signal.to(F64).reshape(signal.shape[0], 1, -1)).permute(2, 0, 1)
    return _grads(y, dy.to(F64), ps)


def conv_stem_backward_matched(signal, w1, b1, w2, b2, w3, b3, dy, w3_t=None, rounded=True):
    """The stem's backward as the kernels compute it: conv3 as an im2col GEMM whose rows (the conv2 output) are fp16, the
    gradient w.r.t. conv3's pre-activation and w.r.t. the rows rounded to bf16, dW3 from the rows rounded to bf16; conv2 and
    conv1 exactly.  w3: conv3's weight in the forward, w3_t: in the backward's transposed copy (default w3).  Same
    arguments and results as conv_stem_backward; with rounded=False it is the exact backward."""
    r16 = (lambda t: t.half().to(F64)) if rounded else (lambda t: t)
    rbf = (lambda t: t.bfloat16().to(F64)) if rounded else (lambda t: t)
    w1, b1, w2, b2 = (t.to(F64).detach().requires_grad_() for t in (w1, b1, w2, b2))
    w3, b3, dy = w3.to(F64), b3.to(F64), dy.to(F64)
    w3_t = w3 if w3_t is None else w3_t.to(F64)
    x = signal.to(F64).reshape(signal.shape[0], 1, -1)
    a1 = bo.swish(torch.nn.functional.conv1d(x, w1, b1, padding=2))
    a2 = bo.swish(torch.nn.functional.conv1d(a1, w2, b2, padding=2))
    cols = torch.nn.functional.pad(a2, (9, 9)).unfold(2, w3.shape[-1], 5)         # (N, 16, T, 19)
    c16 = r16(cols.detach())
    pre = torch.einsum('nctw,ocw->tno', c16, w3) + b3
    sg = torch.sigmoid(pre)
    dpre = rbf(dy * sg * (1 + pre * (1 - sg)))
    dw3 = torch.einsum('tno,nctw->ocw', dpre, rbf(c16))
    db3 = dpre.sum((0, 1))
    dcols = rbf(torch.einsum('tno,ocw->nctw', dpre, w3_t))
    return _grads(cols, dcols, [w1, b1, w2, b2]) + [dw3, db3]


# ----------------------------------------------------------------------------------------------------------- LSTM layer
def lstm_backward(x, w_ih, w_hh, b, dy, reverse):
    """Autograd through bo.lstm_layer (torch.nn.LSTM semantics, either direction) in float64.
    x (T, N, 768), b = b_ih + b_hh, dy (T, N, 768) -> (y, dw_ih, dw_hh, db, dx)."""
    x, w_ih, w_hh, b = (t.to(F64).detach().requires_grad_() for t in (x, w_ih, w_hh, b))
    y = bo.lstm_layer(x, w_ih, w_hh, b, torch.zeros_like(b), reverse)
    dw_ih, dw_hh, db, dx = _grads(y, dy.to(F64), [w_ih, w_hh, b, x])
    return y.detach(), dw_ih, dw_hh, db, dx


def _h_prev(y, reverse):
    """(T, N, H): the hidden state each step of the forward started from (zero for its first step)."""
    z = torch.zeros_like(y[:1])
    return torch.cat([y[1:], z]) if reverse else torch.cat([z, y[:-1]])


def lstm_backward_matched(x, y, w_ih, w_hh, b, dy, reverse, w_ih_t=None, w_hh_t=None, rounded=True):
    """The LSTM layer's backward as the kernels compute it, teacher-forced on the layer's forward output y.

    x (T, N, 768) input, y (T, N, 768) output of the forward (the values the next layer and dW_hh read), w_ih / w_hh the
    forward weights, b = b_ih + b_hh, dy (T, N, 768) gradient w.r.t. y.  w_ih_t / w_hh_t: the weights of the backward's
    transposed copies (default: the forward weights).  With rounded=True the values are rounded where the kernels round:
    the saved gates i, f, g, o and the cell state c to fp16; dz and the outgoing dy to bf16; the transposed x and y copies
    from fp16 to bf16 (and the weights as given).  Returns (dw_ih, dw_hh, db, dx), float64."""
    T, N, _ = x.shape
    H = w_hh.shape[1]
    x, y, w_ih, w_hh, b, dy = (t.to(F64) for t in (x, y, w_ih, w_hh, b, dy))
    w_ih_t = w_ih if w_ih_t is None else w_ih_t.to(F64)
    w_hh_t = w_hh if w_hh_t is None else w_hh_t.to(F64)
    r16 = (lambda t: t.half().to(F64)) if rounded else (lambda t: t)
    rbf = (lambda t: t.bfloat16().to(F64)) if rounded else (lambda t: t)
    hp = _h_prev(y, reverse)
    z = x @ w_ih.t() + b + hp @ w_hh.t()
    zi, zf, zg, zo = z.split(H, dim=2)
    gi, gf, gg, go = torch.sigmoid(zi), torch.sigmoid(zf), torch.tanh(zg), torch.sigmoid(zo)
    order = list(range(T - 1, -1, -1)) if reverse else list(range(T))
    c = torch.empty_like(gi)
    cp = torch.zeros_like(gi[0])
    for t in order:
        cp = gf[t] * cp + gi[t] * gg[t]
        c[t] = cp
    gi, gf, gg, go, c = (r16(t) for t in (gi, gf, gg, go, c))
    c_prev = _h_prev(c, reverse)
    dz = torch.empty(T, N, 4 * H, dtype=F64, device=x.device)
    dc_in = torch.zeros_like(gi[0])
    dz_next = None
    for t in reversed(order):
        dh = dy[t] if dz_next is None else dy[t] + dz_next @ w_hh_t
        tc = torch.tanh(c[t])
        dc = dh * go[t] * (1 - tc * tc) + dc_in
        dzo = dh * tc * go[t] * (1 - go[t])
        dzi = dc * gg[t] * gi[t] * (1 - gi[t])
        dzg = dc * gi[t] * (1 - gg[t] * gg[t])
        dzf = dc * c_prev[t] * gf[t] * (1 - gf[t])
        dc_in = dc * gf[t]
        dz_next = rbf(torch.cat([dzi, dzf, dzg, dzo], dim=1))
        dz[t] = dz_next
    dz2 = dz.reshape(T * N, 4 * H)
    dw_ih = dz2.t() @ rbf(x).reshape(T * N, -1)
    dw_hh = dz2.t() @ rbf(hp).reshape(T * N, -1)
    db = dz2.sum(0)
    dx = rbf(dz @ w_ih_t)
    return dw_ih, dw_hh, db, dx
