"""Layer classes of the encoder under the reference's registry names and constructor arguments
(ub-bonito/bonito/nn.py): `layers` / `register` (:10-16), Swish (:22-24), Serial (:27-36), Reverse (:39-54),
Convolution (:57-84), LinearCRFEncoder (:87-153), Permute (:156-167), LSTM / RNNWrapper (:176-235),
to_dict / from_dict (:238-259).

Parameters are ordinary torch Parameters with the reference's names (conv.weight, rnn.weight_ih_l0,
linear.weight ...), so reference checkpoints load unchanged; the arithmetic runs in libxna_b200.so:

  Serial.forward   recognises [Convolution(1,4,5) Convolution(4,16,5) Convolution(16,768,19,s5) Permute(2,0,1)]
                   (with or without rnn_encoder's drop_rate_bottom Dropouts between them) and runs it as the fused
                   stem (xb_conv_stem_fwd), then LSTM layers (xb_lstm_fwd) and the CRF head (xb_crf_head_fwd);
                   activations stay 16-bit (T, N, 768) on the device in between.  In training the whole encoder is
                   one fused step (xb_encoder_fwd_train[_dropout] / xb_encoder_bwd), dropout included.
  LSTM.forward     one layer on a (T, N, 768) CUDA tensor; `reverse` walks time backwards by indexing.
  LinearCRFEncoder.forward   scale * tanh(x W^T + b) with the blank score expanded in the epilogue -> fp32.

There is no CPU or eager-PyTorch fallback: tensors must live on an sm_100a device, and shapes outside the
sup@v3.3 architecture (features 768, stem 1->4->16->768) raise.
"""
import torch
from torch.nn import Module
from torch.nn.init import orthogonal_

from .engine import Engine

layers = {}

FEATURES = 768


def register(cls):
    """Class decorator: file `cls` in the registry under its lower-cased class name (the `type` of config dicts)."""
    key = cls.__name__.lower()
    cls.name = key
    layers[key] = cls
    return cls


for _activation in (torch.nn.ReLU, torch.nn.Tanh):
    register(_activation)


@register
class Swish(torch.nn.SiLU):
    """x * sigmoid(x); the name the reference's configs use for SiLU."""


def _activation_from(spec):
    """Registry name -> fresh module; anything else (None, a module) is passed through."""
    return layers[spec]() if spec in layers else spec


def _name_of(activation):
    return activation.name if activation else None


def _weights(weight, bias, w_key='W', b_key='b'):
    return {w_key: weight, b_key: [] if bias is None else bias}


def _engine_of(module):
    eng = getattr(module, '_xb_engine', None)
    if eng is None:
        eng = Engine()
        object.__setattr__(module, '_xb_engine', eng)
    return eng


def _adopt(module, engine, slot_counter):
    """Hand `engine` down a module tree and number the LSTM layers (their weight slot in the handle)."""
    object.__setattr__(module, '_xb_engine', engine)
    if isinstance(module, LSTM):
        object.__setattr__(module, '_xb_slot', slot_counter[0])
        slot_counter[0] += 1
    for child in module.children():
        _adopt(child, engine, slot_counter)


def _is_bf16(module):
    p = next(module.parameters(), None)
    return p is not None and p.dtype == torch.bfloat16


@register
class Serial(torch.nn.Sequential):

    def __init__(self, sublayers):
        if isinstance(sublayers, dict):      # slicing a Sequential re-enters here with an OrderedDict:
            super().__init__(sublayers)      # a view of modules that keep their engine and weight slots
            first = next(iter(sublayers.values()), None)
            object.__setattr__(self, '_xb_engine', getattr(first, '_xb_engine', None))
            return
        super().__init__(*sublayers)
        head = next((m for m in self.modules() if isinstance(m, LinearCRFEncoder)), None)
        if head is not None:
            eng = Engine('N' + 'ACGTXYZWVU'[:head.n_base], head.state_len)
        else:
            eng = Engine()
        _adopt(self, eng, [0])

    def set_engine(self, engine):
        _adopt(self, engine, [0])

    def _stem_end(self):
        """Index past the Permute when the leading modules, Dropouts skipped, are the sup@v3.3 convolution stem, else None."""
        mods = list(self)
        core = [i for i, m in enumerate(mods) if not isinstance(m, torch.nn.Dropout)][:4]
        if len(core) < 4:
            return None
        c1, c2, c3, pm = (mods[i] for i in core)
        if not (isinstance(c1, Convolution) and isinstance(c2, Convolution) and isinstance(c3, Convolution)
                and isinstance(pm, Permute)):
            return None
        want = [(1, 4, 5, 1, 2), (4, 16, 5, 1, 2), (16, FEATURES, 19, 5, 9)]
        for c, w in zip((c1, c2, c3), want):
            got = (c.conv.in_channels, c.conv.out_channels, c.conv.kernel_size[0], c.conv.stride[0], c.conv.padding[0])
            if got != w or not isinstance(c.activation, Swish) or c.conv.bias is None:
                return None
        if list(pm.dims) != [2, 0, 1]:
            return None
        return core[3] + 1

    def _stem(self):
        """The three convolutions when the leading modules, Dropouts skipped, are the sup@v3.3 convolution stem, else None.
        Dropout is the identity outside training, so every inference route runs such a model unchanged."""
        end = self._stem_end()
        if end is None:
            return None
        c1, c2, c3 = [m for m in list(self)[:end] if isinstance(m, Convolution)]
        return c1, c2, c3

    def _training_layout(self):
        """(stem, five LSTMs, head, p) when this is the whole sup@v3.3 encoder -- the layout the fused training step
        (xb_encoder_fwd_train_dropout / xb_encoder_bwd) is built for -- else None.  p lists the dropout probabilities of the
        seven places rnn_encoder(drop_rate_bottom=...) puts a torch.nn.Dropout: after each convolution and after LSTM
        layers 0-3 (0.0 where there is none, or where the module is in eval mode).  A Dropout with p > 0 anywhere else
        makes the layout unknown; one with p == 0 is the identity and may stand anywhere."""
        core, drops = [], []                 # modules other than Dropout; the active Dropout after each of them
        for m in self:
            if isinstance(m, torch.nn.Dropout):
                p = float(m.p) if m.training else 0.0
                if p == 0.0:
                    continue
                if not core or drops[-1] is not None:
                    return None
                drops[-1] = p
            else:
                core.append(m)
                drops.append(None)
        if self._stem() is None or len(core) != 10:
            return None
        stem, mods = self._stem(), core[4:]
        if not all(isinstance(m, LSTM) for m in mods[:5]) or not isinstance(mods[5], LinearCRFEncoder):
            return None
        if [m.reverse for m in mods[:5]] != [True, False, True, False, True]:
            return None
        head = mods[5]
        if head.extra_linear or not head.expand_blanks or head.blank_score is None or head.linear.bias is None:
            return None
        if any(drops[i] is not None for i in (3, 8, 9)):     # after the Permute, after LSTM layer 4, after the head
            return None
        p = [drops[i] or 0.0 for i in (0, 1, 2, 4, 5, 6, 7)]
        return stem, mods[:5], head, p

    def forward(self, x):
        mods = list(self)
        stem = self._stem()
        start = 0
        if self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # the training step (bonito/training.py:91-117, after model.train()): one fused forward that keeps the backward's
            # inputs, and an autograd node whose backward is xb_encoder_bwd.  In eval mode (load_model, the basecaller) the
            # layers run the inference kernels and no graph is recorded.
            layout = self._training_layout()
            if layout is None or x.dim() != 3 or x.shape[1] != 1:
                raise RuntimeError('gradients are implemented for the whole sup@v3.3 encoder (conv stem, five LSTMs in the '
                                   'reference directions, LinearCRFEncoder with expand_blanks, dropout only where '
                                   'rnn_encoder(drop_rate_bottom=...) puts it); run other layouts under torch.no_grad()')
            head = layout[2]
            if head.dropout.training and head.dropout.p > 0:
                # where the head applies its dropout in the forward is not recorded in this repository: refuse, do not guess
                raise RuntimeError('LinearCRFEncoder(drop_rate > 0) has no B200 training path; train with drop_rate = 0')
            return _encoder_train_forward(self, layout, x)
        if stem is not None and x.dim() == 3 and x.shape[1] == 1:
            start = self._stem_end()
            for m in mods[:start]:
                if isinstance(m, torch.nn.Dropout) and m.training and m.p > 0:
                    raise RuntimeError('dropout is not part of the B200 forward path; call model.eval()')
            x = _conv_stem_forward(self, stem, x)
        for m in mods[start:]:
            if isinstance(m, torch.nn.Dropout):
                if m.training and m.p > 0:
                    raise RuntimeError('dropout is not part of the B200 forward path; call model.eval()')
                continue
            x = m(x)
        return x

    def sync_weights(self, handle=None):
        """Push every parameter of the tree whose storage changed into the engine's handle."""
        eng = _engine_of(self)
        stem = self._stem()
        if stem is not None:
            _sync_stem(eng, stem)
        for m in self.modules():
            if isinstance(m, (LSTM, LinearCRFEncoder)):
                m._sync(eng)

    def to_dict(self, include_weights=False):
        return {'sublayers': [to_dict(layer, include_weights) for layer in self._modules.values()]}


class _EncoderTrain(torch.autograd.Function):
    """scores = encoder(x) with a backward that fills the gradients of the 28 parameter tensors (xb_encoder_bwd)."""

    @staticmethod
    def forward(ctx, x, handle, dropout_p, seed, *params):
        ctx.handle, ctx.dtypes = handle, [p.dtype for p in params]
        return handle.encoder_train(x, dropout_p=dropout_p, seed=seed)

    @staticmethod
    def backward(ctx, dscores):
        grads = ctx.handle.encoder_backward(dscores)      # the handle replays the masks of its last forward
        return (None, None, None, None) + tuple(grads[k].to(dt) for k, dt in zip(ctx.handle.WEIGHT_KEYS, ctx.dtypes))


def _encoder_train_forward(owner, layout, x):
    stem, lstms, head, dropout_p = layout
    eng = _engine_of(owner)
    N, _, L = x.shape
    if L % 5:
        raise ValueError('chunk length %d is not a multiple of the stride 5' % L)
    h = eng.get(x.device, N, L // 5, bf16=_is_bf16(owner), train=True)
    owner.sync_weights(h)
    params = [t for c in stem for t in (c.conv.weight, c.conv.bias)]
    for m in lstms:
        params += [m.rnn.weight_ih_l0, m.rnn.weight_hh_l0, m.rnn.bias_ih_l0, m.rnn.bias_hh_l0]
    params += [head.linear.weight, head.linear.bias]
    seed = None
    if any(dropout_p):
        # one 63-bit seed per forward from torch's default CPU generator: torch.manual_seed makes the masks repeatable.
        # Without dropout nothing is drawn, so torch's random stream is the same as without this feature.
        seed = int(torch.empty((), dtype=torch.int64).random_().item())
    else:
        dropout_p = None
    return _EncoderTrain.apply(x, h, dropout_p, seed, *params)


def _sync_stem(eng, stem):
    tensors = [t for c in stem for t in (c.conv.weight, c.conv.bias)]
    eng.sync('conv', tensors, lambda hd: hd.load_conv_weights(*tensors))


def _conv_stem_forward(owner, stem, x):
    eng = _engine_of(owner)
    N, _, L = x.shape
    if L % 5:
        raise ValueError('chunk length %d is not a multiple of the stride 5' % L)
    h = eng.get(x.device, N, L // 5, bf16=_is_bf16(owner))
    _sync_stem(eng, stem)
    return h.conv_stem(x)


@register
class Reverse(Module):

    def __init__(self, sublayers):
        super().__init__()
        wrapped = sublayers
        if isinstance(wrapped, list):
            wrapped = Serial(wrapped)
        self.layer = wrapped

    def forward(self, x):
        inner = self.layer
        if isinstance(inner, LSTM):                 # direction by indexing, no flips
            return inner(x, reverse=not inner.reverse)
        return inner(x.flip(0)).flip(0)

    def to_dict(self, include_weights=False):
        inner = self.layer
        return inner.to_dict(include_weights) if isinstance(inner, Serial) else {'sublayers': to_dict(inner, include_weights)}


@register
class Convolution(Module):

    def __init__(self, insize, size, winlen, stride=1, padding=0, bias=True, activation=None):
        super().__init__()
        self.activation = _activation_from(activation)
        self.conv = torch.nn.Conv1d(in_channels=insize, out_channels=size, kernel_size=winlen, stride=stride,
                                    padding=padding, bias=bias)

    def forward(self, x):
        raise RuntimeError(
            'xna_basecaller_b200.nn.Convolution only runs as part of the fused stem '
            'Serial([Convolution(1,4,5), Convolution(4,16,5), Convolution(16,768,19,stride=5), Permute([2,0,1]), ...]); '
            'there is no stand-alone or CPU convolution on this path')

    def to_dict(self, include_weights=False):
        c = self.conv
        (winlen,), (stride,), (padding,) = c.kernel_size, c.stride, c.padding
        out = dict(insize=c.in_channels, size=c.out_channels, bias=c.bias is not None, winlen=winlen, stride=stride,
                   padding=padding, activation=_name_of(self.activation))
        if include_weights:
            out['params'] = _weights(c.weight, c.bias)
        return out


@register
class LinearCRFEncoder(Module):

    def __init__(self, insize, n_base, state_len, bias=True, scale=None, activation=None, blank_score=None,
                 expand_blanks=True, extra_linear=False, drop_rate=0):
        super().__init__()
        self.n_base, self.state_len = n_base, state_len
        self.scale, self.blank_score, self.expand_blanks = scale, blank_score, expand_blanks
        # a learnt blank column per state unless the blank score is a constant: C * (n + 1) or C * n outputs
        states = n_base ** state_len
        width = states * n_base if blank_score is not None else states * (n_base + 1)
        self.extra_linear = extra_linear
        if extra_linear:
            self.linear_ext = torch.nn.Linear(insize, insize, bias=bias)
        self.dropout = torch.nn.Dropout(p=drop_rate)
        self.linear = torch.nn.Linear(insize, width, bias=bias)
        self.activation = _activation_from(activation)

    def forward(self, x):
        if self.extra_linear:
            raise RuntimeError('extra_linear heads have no B200 kernel (the sup@v3.3 models do not use them)')
        if self.dropout.training and self.dropout.p > 0:
            raise RuntimeError('dropout is not part of the B200 forward path; call model.eval()')
        if not isinstance(self.activation, torch.nn.Tanh) or self.blank_score is None:
            raise RuntimeError('the B200 CRF head computes scale*tanh(.) with a constant blank score '
                               '(activation="tanh", blank_score set), as in the sup@v3.3 config')
        if self.linear.in_features != FEATURES:
            raise RuntimeError('the B200 CRF head is built for %d input features' % FEATURES)
        eng = _engine_of(self)
        T, N, _ = x.shape
        h = eng.get(x.device, N, T, bf16=_is_bf16(self))
        self._sync(eng)
        return h.crf_head(x.to(h.dtype16), expand_blanks=self.expand_blanks)

    def _sync(self, eng):
        h = eng.handle
        if h.n_base != self.n_base or h.state_len != self.state_len:
            raise RuntimeError('engine alphabet (n_base %d, state_len %d) does not match the head (%d, %d)'
                               % (h.n_base, h.state_len, self.n_base, self.state_len))
        tensors = [self.linear.weight, self.linear.bias]
        key = (self.scale, self.blank_score, self.expand_blanks)
        eng.sync(('head', key), tensors, lambda hd: hd.load_head_weights(
            self.linear.weight, self.linear.bias, self.scale, self.blank_score, self.expand_blanks))

    def to_dict(self, include_weights=False):
        lin = self.linear
        out = dict(insize=lin.in_features, n_base=self.n_base, state_len=self.state_len, bias=lin.bias is not None,
                   scale=self.scale, activation=_name_of(self.activation), blank_score=self.blank_score)
        if include_weights:
            out['params'] = _weights(lin.weight, lin.bias)
            if self.extra_linear:
                out['params'].update(_weights(self.linear_ext.weight, self.linear_ext.bias, 'W_ext', 'b_ext'))
        return out


@register
class Permute(Module):

    def __init__(self, dims):
        super().__init__()
        self.dims = dims

    def extra_repr(self):
        return 'dims=%s' % (list(self.dims),)

    def forward(self, x):
        return torch.permute(x, tuple(self.dims))

    def to_dict(self, include_weights=False):
        return dict(dims=self.dims)


def truncated_normal(size, dtype=torch.float32, device=None, num_resample=5):
    """Standard normal samples restricted to (-2, 2) (nn.py:170-173 draws `num_resample` candidates per element and keeps
    the first inside the interval; torch's trunc_normal_ samples the same distribution directly)."""
    out = torch.empty(tuple(size), dtype=dtype, device=device)
    return torch.nn.init.trunc_normal_(out, mean=0.0, std=1.0, a=-2.0, b=2.0)


class RNNWrapper(Module):
    """Holds a torch.nn RNN module for its parameters and initialisation (orthogonal weights, truncated-normal
    bias_ih, frozen zero bias_hh: nn.py:195-213); forward goes to the persistent tcgen05 kernel."""

    def __init__(self, rnn_type, *args, reverse=False, orthogonal_weight_init=True, disable_state_bias=True,
                 bidirectional=False, **kwargs):
        super().__init__()
        if bidirectional and reverse:
            raise Exception("'reverse' and 'bidirectional' should not both be set to True")
        self.rnn = rnn_type(*args, bidirectional=bidirectional, **kwargs)
        self.reverse = reverse
        self.init_orthogonal(orthogonal_weight_init)
        self.init_biases()
        if disable_state_bias:
            self.disable_state_bias()

    def _params_named(self, fragments):
        """Parameters of the wrapped RNN whose name contains one of `fragments`."""
        return [(n, q) for n, q in self.rnn.named_parameters() if any(f in n for f in fragments)]

    def forward(self, x, reverse=None):
        rnn = self.rnn
        if not isinstance(rnn, torch.nn.LSTM) or rnn.bidirectional or rnn.num_layers != 1 \
                or rnn.hidden_size != FEATURES or rnn.input_size != FEATURES:
            raise RuntimeError('the B200 recurrent kernel is a single-layer unidirectional LSTM(768, 768)')
        eng = _engine_of(self)
        T, N, _ = x.shape
        h = eng.get(x.device, N, T, bf16=_is_bf16(self))
        self._sync(eng)
        return h.lstm(getattr(self, '_xb_slot', 0), x.to(h.dtype16), self.reverse if reverse is None else reverse)

    def _sync(self, eng):
        rnn = self.rnn
        slot = getattr(self, '_xb_slot', 0)
        if slot >= 5:
            raise RuntimeError('the engine holds five LSTM weight slots; layer %d does not fit' % slot)
        w = [rnn.weight_ih_l0, rnn.weight_hh_l0, rnn.bias_ih_l0, rnn.bias_hh_l0]
        eng.sync(('lstm', slot), w, lambda hd: hd.load_lstm_weights(slot, *w))

    def init_biases(self, types=('bias_ih',)):
        """Input biases ~ 0.5 * N(0, 1) truncated to (-2, 2) (nn.py:195-199)."""
        with torch.no_grad():
            for _, q in self._params_named(types):
                q.copy_(truncated_normal(q.shape, dtype=q.dtype, device=q.device).mul_(0.5))

    def init_orthogonal(self, types=True):
        """Every (hidden x in) gate block of the selected weight matrices gets its own orthogonal init (nn.py:201-207)."""
        if types is True:
            types = ('weight_ih', 'weight_hh')
        if not types:
            return
        H = self.rnn.hidden_size
        for _, q in self._params_named(types):
            for gate_block in q.split(H, dim=0):
                orthogonal_(gate_block)

    def disable_state_bias(self):
        """bias_hh is frozen at zero: only bias_ih is learnt, but the parameter stays in the state_dict (nn.py:209-213)."""
        for _, q in self._params_named(('bias_hh',)):
            q.requires_grad_(False)
            with torch.no_grad():
                q.zero_()


@register
class LSTM(RNNWrapper):

    def __init__(self, size, insize, bias=True, reverse=False):
        super().__init__(torch.nn.LSTM, size, insize, bias=bias, reverse=reverse)

    def to_dict(self, include_weights=False):
        r = self.rnn
        out = dict(size=r.hidden_size, insize=r.input_size, bias=r.bias, reverse=self.reverse)
        if include_weights:       # per-gate views: input weights, state weights, input bias (bias_hh is identically zero)
            out['params'] = dict(iW=r.weight_ih_l0.view(4, r.hidden_size, r.input_size),
                                 sW=r.weight_hh_l0.view(4, r.hidden_size, r.hidden_size),
                                 b=r.bias_ih_l0.view(4, r.hidden_size))
        return out


def to_dict(layer, include_weights=False):
    """{'type': registry name, **the layer's own description}."""
    described = layer.to_dict(include_weights) if hasattr(layer, 'to_dict') else {}
    return dict(type=layer.name, **described)


def from_dict(model_dict, layer_types=None):
    """Inverse of to_dict: build the module tree a (new-style) config describes."""
    registry = layers if layer_types is None else layer_types
    kwargs = {k: v for k, v in model_dict.items() if k != 'type'}
    cls = registry[model_dict['type']]
    nested = kwargs.get('sublayers')
    if isinstance(nested, list):
        kwargs['sublayers'] = [from_dict(d, registry) for d in nested]
    elif nested is not None:
        kwargs['sublayers'] = from_dict(nested, registry)
    try:
        return cls(**kwargs)
    except Exception as e:
        raise Exception('Failed to build layer of type %s with args %s' % (cls, kwargs)) from e
