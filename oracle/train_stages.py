"""float64 references of the three stages of the encoder backward (xb_encoder_bwd_stages): the CRF head, one LSTM layer
and the convolution stem.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

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
