"""ctypes binding of libxna_b200.so (include/xna_basecaller.h) + a thin torch-tensor front end.

There is no CPU fallback: if the shared library is missing, or no sm_100 GPU is present, every
compute entry point raises.  torch is used only for device memory and streams.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libxna_b200.so')

XB_FLAG_BF16 = 1
XB_FLAG_NO_ENCODER = 2
XB_FLAG_TRAIN = 8
XB_SIG_F32, XB_SIG_F16, XB_SIG_I16 = 0, 1, 2
NUM_WEIGHTS = 28
DROPOUT_SITES = 7       # conv1, conv2, conv3 outputs, outputs of LSTM layers 0..3 (XB_DROPOUT_SITES)

# every symbol include/xna_basecaller.h declares (tests check that the library exports them all)
SYMBOLS = (
    'xb_abi_version', 'xb_last_error', 'xb_create', 'xb_destroy', 'xb_load_weights', 'xb_load_conv_weights',
    'xb_load_lstm_weights', 'xb_load_head_weights', 'xb_conv_stem_fwd',
    'xb_lstm_fwd', 'xb_lstm_stack_fwd', 'xb_crf_head_fwd', 'xb_encoder_fwd', 'xb_crf_logz',
    'xb_crf_forward_scores', 'xb_crf_backward_scores', 'xb_crf_posteriors', 'xb_crf_viterbi', 'xb_crf_decode',
    'xb_ctc_crf_loss_fwd', 'xb_ctc_crf_loss_bwd', 'xb_stitch', 'xb_gather_chunks', 'xb_preprocess_reads', 'xb_compute_scores_host', 'xb_compute_scores_submit', 'xb_compute_scores_wait', 'xb_launch_count', 'xb_gemm_selftest',
    'xb_set_profiling', 'xb_stage_times', 'xb_crf_head_fwd_exp', 'xb_crf_decode_exp', 'xb_basecall_chunks',
    'xb_crf_logz_s', 'xb_crf_forward_scores_s', 'xb_crf_backward_scores_s', 'xb_crf_posteriors_max',
    'xb_encoder_fwd_train', 'xb_encoder_bwd', 'xb_adamw_step', 'xb_crf_beam_search',
    'xb_align_counts', 'xb_encoder_fwd_train_dropout', 'xb_dropout_keep',
)
STAGES = ('conv12_im2col', 'conv3_gemm', 'lstm_inproj_gemm', 'lstm_recurrence', 'crf_head_gemm', 'crf_alpha',
          'crf_backward', 'crf_viterbi', 'train_bptt', 'train_transpose', 'train_weight_grad_gemm', 'train_input_grad_gemm', 'train_head_conv_bwd')

_lib = None


def load():
    """dlopen the library (works without a GPU; compute calls do not)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'xna_basecaller_b200: %s is missing -- build it with `python -m xna_basecaller_b200.build` '
            '(there is no CPU or PyTorch fallback for this path)' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, ci, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    lib.xb_abi_version.restype = ci
    lib.xb_last_error.restype = ctypes.c_char_p
    lib.xb_last_error.argtypes = [vp]
    lib.xb_create.argtypes = [ctypes.POINTER(vp), ci, ci, ci, ci, ci, ctypes.c_char_p, ci]
    lib.xb_destroy.argtypes = [vp]
    lib.xb_load_weights.argtypes = [vp, ctypes.POINTER(vp), ci, cf, cf, ci, vp]
    lib.xb_load_conv_weights.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.xb_load_lstm_weights.argtypes = [vp, ci, vp, vp, vp, vp, vp]
    lib.xb_load_head_weights.argtypes = [vp, vp, vp, cf, cf, ci, vp]
    lib.xb_conv_stem_fwd.argtypes = [vp, vp, ci, ci, ci, vp, vp]
    lib.xb_lstm_fwd.argtypes = [vp, ci, vp, vp, ci, ci, ci, vp]
    lib.xb_lstm_stack_fwd.argtypes = [vp, vp, vp, ci, ci, vp]
    lib.xb_crf_head_fwd.argtypes = [vp, vp, vp, ci, ci, vp]
    lib.xb_encoder_fwd.argtypes = [vp, vp, ci, ci, ci, vp, vp]
    lib.xb_crf_logz.argtypes = [vp, vp, ci, ci, vp, vp]
    lib.xb_crf_forward_scores.argtypes = [vp, vp, ci, ci, vp, vp]
    lib.xb_crf_backward_scores.argtypes = [vp, vp, ci, ci, vp, vp]
    lib.xb_crf_posteriors.argtypes = [vp, vp, ci, ci, vp, vp]
    lib.xb_encoder_fwd_train.argtypes = [vp, vp, ci, ci, ci, vp, vp]
    lib.xb_encoder_bwd.argtypes = [vp, vp, ci, vp, vp, ctypes.POINTER(vp), ci, vp]
    lib.xb_encoder_fwd_train_dropout.argtypes = [vp, vp, ci, ci, ci, ctypes.POINTER(cf), ctypes.c_uint64, vp, vp]
    lib.xb_dropout_keep.argtypes = [ctypes.c_uint64, ci, cf, ctypes.c_int64, vp, vp]
    lib.xb_adamw_step.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp),
                                  ctypes.POINTER(ctypes.c_int64), ci, cf, cf, cf, cf, cf, cf, ctypes.c_int64, vp, vp, vp]
    lib.xb_align_counts.argtypes = [vp, ci, vp, vp, ci, vp, ci, vp, vp]
    lib.xb_crf_beam_search.argtypes = [vp, vp, ci, ci, ci, cf, vp, vp, vp, vp, vp]
    lib.xb_crf_logz_s.argtypes = [vp, vp, ci, ci, ci, vp, vp]
    lib.xb_crf_forward_scores_s.argtypes = [vp, vp, ci, ci, ci, vp, vp]
    lib.xb_crf_backward_scores_s.argtypes = [vp, vp, ci, ci, ci, vp, vp]
    lib.xb_crf_posteriors_max.argtypes = [vp, vp, ci, ci, vp, vp, vp]
    lib.xb_crf_viterbi.argtypes = [vp, vp, ci, ci, vp, vp]
    lib.xb_crf_decode.argtypes = [vp, vp, ci, ci, vp, vp, vp, vp, vp, vp]
    lib.xb_crf_decode_exp.argtypes = [vp, vp, ci, ci, vp, vp, vp, vp, vp, vp]
    lib.xb_crf_head_fwd_exp.argtypes = [vp, vp, vp, ci, ci, vp]
    lib.xb_basecall_chunks.argtypes = [vp, vp, ci, ci, ci, vp, vp, vp, vp]
    lib.xb_ctc_crf_loss_fwd.argtypes = [vp, vp, ci, ci, vp, ci, vp, ci, vp, vp]
    lib.xb_compute_scores_submit.argtypes = [vp, ci, vp, ci, ci, vp, vp, vp]
    lib.xb_compute_scores_wait.argtypes = [vp, ci]
    lib.xb_preprocess_reads.argtypes = [vp, vp, vp, vp, vp, vp, ci, vp, vp, vp, vp]
    lib.xb_ctc_crf_loss_bwd.argtypes = [vp, vp, ci, ci, vp, ci, vp, ci, vp, vp, vp, vp]
    lib.xb_stitch.argtypes = [vp, vp, ci, vp, vp, vp, ci, ci, ci, ci, ci, vp, ci, vp, vp]
    lib.xb_gather_chunks.argtypes = [vp, vp, ci, vp, vp, vp, vp, ci, ci, vp, vp]
    lib.xb_compute_scores_host.argtypes = [vp, vp, ci, ci, vp, vp, vp]
    lib.xb_launch_count.restype = ctypes.c_int64
    lib.xb_launch_count.argtypes = [vp]
    lib.xb_gemm_selftest.argtypes = [vp, vp, vp, vp, ci, ci, ci, vp]
    lib.xb_set_profiling.argtypes = [vp, ci]
    lib.xb_stage_times.argtypes = [vp, vp, vp]
    for name in SYMBOLS:
        if name not in ('xb_last_error', 'xb_launch_count'):
            getattr(lib, name).restype = ci
    _lib = lib
    return lib


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def align_counts(seq, seq_len, ref, ref_len):
    """xb_align_counts: local alignment counts of seq[p, :seq_len[p]] (query) against ref[p, :ref_len[p]] for every row p.
    seq / ref: (N, *) int8 CUDA tensors with unit column stride (left-packed rows, as the decode writes them); lengths (N,)
    on the same device.  Returns (N, 5) int32 on the device: (score, eq, x, ins, del).  Synchronises the current stream
    once (the library checks the lengths on the host)."""
    if not torch.cuda.is_available():
        raise RuntimeError('xna_basecaller_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    lib = load()
    dev = seq.device
    if dev.type != 'cuda' or ref.device != dev:
        raise ValueError('align_counts takes CUDA tensors on one device')
    if seq.dtype != torch.int8 or ref.dtype != torch.int8 or seq.dim() != 2 or ref.dim() != 2 or len(seq) != len(ref):
        raise ValueError('seq and ref must be (N, *) int8 with the same N')
    if seq.stride(1) != 1:
        seq = seq.contiguous()
    if ref.stride(1) != 1:
        ref = ref.contiguous()
    n = seq.shape[0]
    sl = seq_len.to(dev, torch.int32).contiguous()
    rl = ref_len.to(dev, torch.int32).contiguous()
    if sl.numel() != n or rl.numel() != n:
        raise ValueError('one length per row')
    counts = torch.empty(n, 5, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.xb_align_counts(_ptr(seq), seq.stride(0), _ptr(sl), _ptr(ref), ref.stride(0), _ptr(rl), n, _ptr(counts),
                                 _stream(dev))
    if rc != 0:
        raise RuntimeError('xb_align_counts failed (%d): %s' % (rc, lib.xb_last_error(None).decode()))
    return counts


def dropout_probabilities(p):
    """The XB_DROPOUT_SITES probabilities as a list of floats; ValueError unless there are seven, each 0 <= p < 1."""
    p = [float(v) for v in p]
    if len(p) != DROPOUT_SITES:
        raise ValueError('dropout needs %d probabilities (one per site), got %d' % (DROPOUT_SITES, len(p)))
    for site, v in enumerate(p):
        if not (0.0 <= v < 1.0 and ctypes.c_float(v).value < 1.0):      # the library takes p as a float
            raise ValueError('dropout probability of site %d must lie in [0, 1), got %r' % (site, v))
    return p


def dropout_keep(seed, site, p, n, device=None):
    """xb_dropout_keep: the keep flags (n,) bool on the device of elements 0 .. n-1 of dropout site `site` under (seed, p),
    from the device function the training kernels use."""
    if not torch.cuda.is_available():
        raise RuntimeError('xna_basecaller_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    lib = load()
    if not 0 <= int(site) < DROPOUT_SITES:
        raise ValueError('dropout site %r out of range' % (site,))
    p = dropout_probabilities([p if s == int(site) else 0.0 for s in range(DROPOUT_SITES)])[int(site)]
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    keep = torch.empty(int(n), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.xb_dropout_keep(int(seed) & 0xffffffffffffffff, int(site), float(p), int(n), _ptr(keep), _stream(dev))
    if rc != 0:
        raise RuntimeError('xb_dropout_keep failed (%d): %s' % (rc, lib.xb_last_error(None).decode()))
    return keep.bool()


class Handle:
    """One xb_handle: a device, an alphabet, capacity (max_N chunks x max_T steps) and, after
    load_weights(), the repacked encoder weights."""

    def __init__(self, alphabet, state_len=3, max_N=64, max_T=800, device=0, bf16=False, encoder=True, train=False):
        if not torch.cuda.is_available():
            raise RuntimeError('xna_basecaller_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self.lib = load()
        self.alphabet = ''.join(alphabet)
        self.n_base = len(self.alphabet) - 1
        self.state_len = state_len
        self.C = self.n_base ** state_len
        self.NZ = self.n_base + 1
        self.max_N, self.max_T = max_N, max_T
        self.device = torch.device('cuda', device) if not isinstance(device, torch.device) else device
        self.bf16 = bf16
        self.dtype16 = torch.float16        # activations are fp16 in both modes; bf16 rounds the WEIGHTS to bfloat16
        flags = (XB_FLAG_BF16 if bf16 else 0) | (0 if encoder else XB_FLAG_NO_ENCODER) | (XB_FLAG_TRAIN if train else 0)
        self.train = train
        h = ctypes.c_void_p()
        rc = self.lib.xb_create(ctypes.byref(h), self.device.index or 0, max_N, max_T, self.n_base, state_len,
                                self.alphabet.encode(), flags)
        if rc != 0:
            raise RuntimeError('xb_create failed (%d): %s' % (rc, self.lib.xb_last_error(None).decode()))
        self.h = h
        self._keep = None

    def close(self):
        if getattr(self, 'h', None):
            self.lib.xb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError('%s failed (%d): %s' % (what, rc, self.lib.xb_last_error(self.h).decode()))

    @property
    def launches(self):
        return int(self.lib.xb_launch_count(self.h))

    def set_profiling(self, on):
        self._check(self.lib.xb_set_profiling(self.h, int(on)), 'xb_set_profiling')

    def stage_times(self):
        """{stage: (milliseconds, spans)} accumulated since the last call (CUDA events on the launch stream)."""
        ms = (ctypes.c_float * len(STAGES))()
        n = (ctypes.c_int * len(STAGES))()
        self._check(self.lib.xb_stage_times(self.h, ms, n), 'xb_stage_times')
        return {name: (float(ms[i]), int(n[i])) for i, name in enumerate(STAGES)}

    # ------------------------------------------------------------------ weights / encoder
    def load_weights(self, state_dict, scale=5.0, blank_score=2.0, expand_blanks=True):
        """state_dict with the reference keys (encoder.0.conv.weight ... encoder.9.linear.bias)."""
        keys = []
        for i in range(3):
            keys += ['encoder.%d.conv.weight' % i, 'encoder.%d.conv.bias' % i]
        for i in range(4, 9):
            keys += ['encoder.%d.rnn.%s' % (i, k) for k in ('weight_ih_l0', 'weight_hh_l0', 'bias_ih_l0', 'bias_hh_l0')]
        keys += ['encoder.9.linear.weight', 'encoder.9.linear.bias']
        tensors = [state_dict[k].detach().to(self.device, torch.float32).contiguous() for k in keys]
        arr = (ctypes.c_void_p * NUM_WEIGHTS)(*[t.data_ptr() for t in tensors])
        rc = self.lib.xb_load_weights(self.h, arr, NUM_WEIGHTS, float(scale),
                                      float(blank_score if blank_score is not None else 0.0),
                                      int(bool(expand_blanks) and blank_score is not None), _stream(self.device))
        self._check(rc, 'xb_load_weights')
        torch.cuda.current_stream(self.device).synchronize()   # tensors may be freed after this

    def _f32(self, t):
        return t.detach().to(self.device, torch.float32).contiguous()

    def load_conv_weights(self, w1, b1, w2, b2, w3, b3):
        ts = [self._f32(t) for t in (w1, b1, w2, b2, w3, b3)]
        self._check(self.lib.xb_load_conv_weights(self.h, *[_ptr(t) for t in ts], _stream(self.device)),
                    'xb_load_conv_weights')
        torch.cuda.current_stream(self.device).synchronize()

    def load_lstm_weights(self, layer, w_ih, w_hh, b_ih, b_hh):
        ts = [self._f32(t) for t in (w_ih, w_hh, b_ih, b_hh)]
        self._check(self.lib.xb_load_lstm_weights(self.h, int(layer), *[_ptr(t) for t in ts], _stream(self.device)),
                    'xb_load_lstm_weights')
        torch.cuda.current_stream(self.device).synchronize()

    def load_head_weights(self, w, b, scale=5.0, blank_score=2.0, expand_blanks=True):
        w = self._f32(w)
        b = self._f32(b) if b is not None else None
        self._check(self.lib.xb_load_head_weights(self.h, _ptr(w), _ptr(b), float(scale if scale is not None else 1.0),
                                                  float(blank_score if blank_score is not None else 0.0),
                                                  int(bool(expand_blanks) and blank_score is not None),
                                                  _stream(self.device)), 'xb_load_head_weights')
        torch.cuda.current_stream(self.device).synchronize()

    def _sig(self, signal):
        if signal.dim() == 3:
            signal = signal[:, 0, :]
        signal = signal.contiguous()
        code = {torch.float32: XB_SIG_F32, torch.float16: XB_SIG_F16, torch.int16: XB_SIG_I16}.get(signal.dtype)
        if code is None:
            signal, code = signal.float(), XB_SIG_F32
        return signal, code

    def conv_stem(self, signal):
        signal, code = self._sig(signal.to(self.device))
        N, L = signal.shape
        out = torch.empty(L // 5, N, 768, dtype=self.dtype16, device=self.device)
        self._check(self.lib.xb_conv_stem_fwd(self.h, _ptr(signal), code, N, L, _ptr(out), _stream(self.device)),
                    'xb_conv_stem_fwd')
        return out

    def lstm(self, layer, x, reverse):
        x = x.contiguous()
        T, N, _ = x.shape
        y = torch.empty_like(x)
        self._check(self.lib.xb_lstm_fwd(self.h, layer, _ptr(x), _ptr(y), T, N, int(reverse), _stream(self.device)),
                    'xb_lstm_fwd')
        return y

    def lstm_stack(self, x):
        x = x.contiguous().clone()
        T, N, _ = x.shape
        y = torch.empty_like(x)
        self._check(self.lib.xb_lstm_stack_fwd(self.h, _ptr(x), _ptr(y), T, N, _stream(self.device)), 'xb_lstm_stack_fwd')
        return y

    def crf_head(self, x, expand_blanks=True, exp=False):
        """LinearCRFEncoder scores; exp=True: exp(scores), the hand-over format of the fused route."""
        x = x.contiguous()
        T, N, _ = x.shape
        width = self.C * self.NZ if expand_blanks else self.C * self.n_base
        scores = torch.empty(T, N, width, dtype=torch.float32, device=self.device)
        fn = self.lib.xb_crf_head_fwd_exp if exp else self.lib.xb_crf_head_fwd
        self._check(fn(self.h, _ptr(x), _ptr(scores), T, N, _stream(self.device)), 'xb_crf_head_fwd')
        return scores

    def basecall_chunks(self, signal, want_qstring=False, out=None):
        """Fused encoder + decode of device-resident chunks: (seq (N,T) int8 left-packed, qstring | None, lens (N) int32).
        out: optional contiguous (N, T) int8 device tensor that receives the packed rows."""
        signal, code = self._sig(signal.to(self.device))
        N, L = signal.shape
        T = L // 5
        seq = out if out is not None else torch.empty(N, T, dtype=torch.int8, device=self.device)
        qs = torch.empty(N, T, dtype=torch.int8, device=self.device) if want_qstring else None
        lens = torch.empty(N, dtype=torch.int32, device=self.device)
        self._check(self.lib.xb_basecall_chunks(self.h, _ptr(signal), code, N, L, _ptr(seq), _ptr(qs), _ptr(lens),
                                                _stream(self.device)), 'xb_basecall_chunks')
        return seq, qs, lens

    def encoder(self, signal, expand_blanks=True):
        signal, code = self._sig(signal.to(self.device))
        N, L = signal.shape
        width = self.C * self.NZ if expand_blanks else self.C * self.n_base
        scores = torch.empty(L // 5, N, width, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_encoder_fwd(self.h, _ptr(signal), code, N, L, _ptr(scores), _stream(self.device)),
                    'xb_encoder_fwd')
        return scores

    # ------------------------------------------------------------------ training step (handle created with train=True)
    WEIGHT_KEYS = (['encoder.%d.conv.%s' % (i, k) for i in range(3) for k in ('weight', 'bias')] +
                   ['encoder.%d.rnn.%s' % (i, k) for i in range(4, 9)
                    for k in ('weight_ih_l0', 'weight_hh_l0', 'bias_ih_l0', 'bias_hh_l0')] +
                   ['encoder.9.linear.weight', 'encoder.9.linear.bias'])

    def encoder_train(self, signal, dropout_p=None, seed=None):
        """Training forward: scores (T, N, C*NZ) fp32; the handle keeps what encoder_backward needs.
        dropout_p: None, or the probabilities of the DROPOUT_SITES dropout sites (xb_encoder_fwd_train_dropout) with the
        64-bit `seed` of their masks; encoder_backward applies the same masks."""
        if dropout_p is not None:
            dropout_p = dropout_probabilities(dropout_p)
            if seed is None:
                raise ValueError('dropout needs a seed')
        signal, code = self._sig(signal.to(self.device))
        N, L = signal.shape
        scores = torch.empty(L // 5, N, self.C * self.NZ, dtype=torch.float32, device=self.device)
        if dropout_p is None:
            self._check(self.lib.xb_encoder_fwd_train(self.h, _ptr(signal), code, N, L, _ptr(scores), _stream(self.device)),
                        'xb_encoder_fwd_train')
        else:
            p = (ctypes.c_float * DROPOUT_SITES)(*dropout_p)
            self._check(self.lib.xb_encoder_fwd_train_dropout(self.h, _ptr(signal), code, N, L, p,
                                                              int(seed) & 0xffffffffffffffff, _ptr(scores),
                                                              _stream(self.device)), 'xb_encoder_fwd_train_dropout')
        self._train_keep = (signal, code, scores)
        return scores

    def encoder_backward(self, dscores):
        """dscores (T, N, C*NZ) fp32 -> {reference state_dict key: fp32 gradient in the reference's layout}."""
        signal, code, scores = self._train_keep
        ds = dscores.to(self.device, torch.float32).contiguous()
        head_rows = self.C * self.n_base
        shapes = [(4, 1, 5), (4,), (16, 4, 5), (16,), (768, 320), (768,)]
        for _ in range(5):
            shapes += [(3072, 768), (3072, 768), (3072,), (3072,)]
        shapes += [(head_rows, 768), (head_rows,)]
        grads = [torch.zeros(*s, dtype=torch.float32, device=self.device) for s in shapes]
        arr = (ctypes.c_void_p * NUM_WEIGHTS)(*[g.data_ptr() for g in grads])
        self._check(self.lib.xb_encoder_bwd(self.h, _ptr(signal), code, _ptr(scores), _ptr(ds), arr, NUM_WEIGHTS,
                                            _stream(self.device)), 'xb_encoder_bwd')
        grads[4] = grads[4][:, :304].reshape(768, 19, 16).permute(0, 2, 1).contiguous()      # [out][tap][in] -> (768, 16, 19)
        return dict(zip(self.WEIGHT_KEYS, grads))

    # ------------------------------------------------------------------ CRF
    def _scores(self, scores):
        s = scores.to(self.device, torch.float32).contiguous()
        T, N, W = s.shape
        if W != self.C * self.NZ:
            raise ValueError('scores last dim %d != C*NZ = %d' % (W, self.C * self.NZ))
        return s, T, N

    def logZ(self, scores, semiring=0):
        """semiring 0 = Log (logsumexp over paths), 1 = Max (score of the best path)."""
        s, T, N = self._scores(scores)
        out = torch.empty(N, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_crf_logz_s(self.h, _ptr(s), T, N, int(semiring), _ptr(out), _stream(self.device)), 'xb_crf_logz_s')
        return out

    def forward_scores(self, scores, semiring=0):
        s, T, N = self._scores(scores)
        out = torch.empty(T + 1, N, self.C, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_crf_forward_scores_s(self.h, _ptr(s), T, N, int(semiring), _ptr(out), _stream(self.device)),
                    'xb_crf_forward_scores_s')
        return out

    def backward_scores(self, scores, semiring=0):
        s, T, N = self._scores(scores)
        out = torch.empty(T + 1, N, self.C, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_crf_backward_scores_s(self.h, _ptr(s), T, N, int(semiring), _ptr(out), _stream(self.device)),
                    'xb_crf_backward_scores_s')
        return out

    def posteriors_max(self, scores, want_onehot=True):
        """posteriors(scores, Max): (edges (N, T) int32 flat arg-max edge index per step, one-hot (T, N, C*NZ) | None)."""
        s, T, N = self._scores(scores)
        edges = torch.empty(N, T, dtype=torch.int32, device=self.device)
        post = torch.empty_like(s) if want_onehot else None
        self._check(self.lib.xb_crf_posteriors_max(self.h, _ptr(s), T, N, _ptr(edges), _ptr(post), _stream(self.device)),
                    'xb_crf_posteriors_max')
        return edges, post

    def posteriors(self, scores):
        s, T, N = self._scores(scores)
        out = torch.empty_like(s)
        self._check(self.lib.xb_crf_posteriors(self.h, _ptr(s), T, N, _ptr(out), _stream(self.device)), 'xb_crf_posteriors')
        return out

    def viterbi(self, scores):
        """labels (N, T) int8."""
        s, T, N = self._scores(scores)
        out = torch.empty(N, T, dtype=torch.int8, device=self.device)
        self._check(self.lib.xb_crf_viterbi(self.h, _ptr(s), T, N, _ptr(out), _stream(self.device)), 'xb_crf_viterbi')
        return out

    def decode(self, scores, want_labels=False, want_post=False, want_qstring=True, exp_input=False):
        """sequence (N,T) int8, qstring (N,T) int8 | None, lens (N) int32 [, labels (N,T)] [, post].
        exp_input: `scores` holds exp(scores) (crf_head(..., exp=True))."""
        s, T, N = self._scores(scores)
        seq = torch.empty(N, T, dtype=torch.int8, device=self.device)
        qs = torch.empty(N, T, dtype=torch.int8, device=self.device) if want_qstring else None
        lens = torch.empty(N, dtype=torch.int32, device=self.device)
        labels = torch.empty(N, T, dtype=torch.int8, device=self.device) if want_labels else None
        post = torch.empty_like(s) if want_post else None
        fn = self.lib.xb_crf_decode_exp if exp_input else self.lib.xb_crf_decode
        self._check(fn(self.h, _ptr(s), T, N, _ptr(seq), _ptr(qs), _ptr(lens), _ptr(labels),
                       _ptr(post), _stream(self.device)), 'xb_crf_decode')
        out = [seq, qs, lens]
        if want_labels:
            out.append(labels)
        if want_post:
            out.append(post)
        return tuple(out)

    def beam_search(self, scores, beam_width=32, beam_cut=100.0):
        """(sequence (N,T) int8 left-packed letters, qstring (N,T) int8 phred+33, moves (N,T) bool, lens (N) int32)."""
        s, T, N = self._scores(scores)
        seq = torch.empty(N, T, dtype=torch.int8, device=self.device)
        qs = torch.empty(N, T, dtype=torch.int8, device=self.device)
        mv = torch.empty(N, T, dtype=torch.int8, device=self.device)
        lens = torch.empty(N, dtype=torch.int32, device=self.device)
        self._check(self.lib.xb_crf_beam_search(self.h, _ptr(s), T, N, int(beam_width), float(beam_cut), _ptr(seq), _ptr(qs),
                                                _ptr(mv), _ptr(lens), _stream(self.device)), 'xb_crf_beam_search')
        return seq, qs, mv.bool(), lens

    def ctc_loss(self, scores, targets, lengths, normalise=True):
        s, T, N = self._scores(scores)
        tg = targets.to(self.device, torch.int32).contiguous()
        ln = lengths.to(self.device, torch.int32).contiguous()
        out = torch.empty(N, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_ctc_crf_loss_fwd(self.h, _ptr(s), T, N, _ptr(tg), tg.shape[1], _ptr(ln),
                                                 int(normalise), _ptr(out), _stream(self.device)), 'xb_ctc_crf_loss_fwd')
        return out

    def ctc_loss_bwd(self, scores, targets, lengths, grad_loss, normalise=True):
        """d(sum_n grad_loss[n] * loss[n]) / d scores, (T, N, C*NZ) fp32."""
        s, T, N = self._scores(scores)
        tg = targets.to(self.device, torch.int32).contiguous()
        ln = lengths.to(self.device, torch.int32).contiguous()
        gl = grad_loss.to(self.device, torch.float32).contiguous()
        npos = tg.shape[1] - (self.state_len - 1)
        ws = torch.empty((T + 1) * N * max(npos, 1), dtype=torch.float32, device=self.device)
        grad = torch.empty_like(s)
        self._check(self.lib.xb_ctc_crf_loss_bwd(self.h, _ptr(s), T, N, _ptr(tg), tg.shape[1], _ptr(ln), int(normalise),
                                                 _ptr(gl), _ptr(ws), _ptr(grad), _stream(self.device)),
                    'xb_ctc_crf_loss_bwd')
        return grad

    def stitch(self, rows, chunk_first, chunk_count, read_len, chunksize, overlap, stride=5, out_stride=None, reverse=False):
        rows = rows.to(self.device, torch.int8).contiguous()
        T = rows.shape[1]
        cf = torch.as_tensor(chunk_first, dtype=torch.int32, device=self.device)
        cc = torch.as_tensor(chunk_count, dtype=torch.int32, device=self.device)
        rl = torch.as_tensor(read_len, dtype=torch.int32, device=self.device)
        n_reads = cf.numel()
        if out_stride is None:
            out_stride = int(cc.max().item()) * T
        out = torch.zeros(n_reads, out_stride, dtype=torch.int8, device=self.device)
        out_len = torch.empty(n_reads, dtype=torch.int32, device=self.device)
        self._check(self.lib.xb_stitch(self.h, _ptr(rows), T, _ptr(cf), _ptr(cc), _ptr(rl), n_reads, chunksize, overlap,
                                       stride, int(bool(reverse)), _ptr(out), out_stride, _ptr(out_len),
                                       _stream(self.device)), 'xb_stitch')
        return out, out_len

    def gather_chunks(self, signal, read_offset, read_len, chunk_read, chunk_start, L, out=None):
        """chunk batch (n_chunks, L) fp32 cut on the device from a resident read set (fp32 or int16)."""
        code = {torch.float32: XB_SIG_F32, torch.int16: XB_SIG_I16}[signal.dtype]
        n = chunk_read.numel()
        if out is None:
            out = torch.empty(n, L, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_gather_chunks(self.h, _ptr(signal), code, _ptr(read_offset), _ptr(read_len), _ptr(chunk_read),
                                              _ptr(chunk_start), n, L, _ptr(out), _stream(self.device)), 'xb_gather_chunks')
        return out

    def preprocess(self, raw, read_offset, read_len, scaling, offset):
        """Raw int16 reads (concatenated) -> (normalised float32 signal in the same layout, out_len (n) int32,
        stats (n, 4) float32 = trim start, med, mad, mode).  fast5.py:88-100 on the GPU."""
        dev = self.device
        raw = raw.to(dev, torch.int16).contiguous()
        ro = torch.as_tensor(read_offset, dtype=torch.int64, device=dev).contiguous()
        rl = torch.as_tensor(read_len, dtype=torch.int32, device=dev).contiguous()
        sc = torch.as_tensor(scaling, dtype=torch.float64, device=dev).contiguous()
        of = torch.as_tensor(offset, dtype=torch.int32, device=dev).contiguous()
        n = ro.numel()
        out = torch.empty(raw.numel(), dtype=torch.float32, device=dev)
        out_len = torch.empty(n, dtype=torch.int32, device=dev)
        stats = torch.empty(n, 4, dtype=torch.float32, device=dev)
        self._check(self.lib.xb_preprocess_reads(self.h, _ptr(raw), _ptr(ro), _ptr(rl), _ptr(sc), _ptr(of), n, _ptr(out),
                                                 _ptr(out_len), _ptr(stats), _stream(dev)), 'xb_preprocess_reads')
        return out, out_len, stats

    def compute_scores_submit(self, slot, signal_host, seq_host, lens_host):
        """Enqueue one batch (pinned host tensors) into slot 0 / 1; results are valid after compute_scores_wait(slot)."""
        N, L = signal_host.shape
        self._check(self.lib.xb_compute_scores_submit(self.h, int(slot), _ptr(signal_host), N, L, _ptr(seq_host),
                                                      _ptr(lens_host), _stream(self.device)), 'xb_compute_scores_submit')

    def compute_scores_wait(self, slot):
        self._check(self.lib.xb_compute_scores_wait(self.h, int(slot)), 'xb_compute_scores_wait')

    def compute_scores_host(self, signal_host, seq_host=None, lens_host=None):
        """signal_host: (N, L) fp32 CPU tensor (pinned for async copies) -> packed sequences on the host."""
        if signal_host.dim() == 3:
            signal_host = signal_host[:, 0, :]
        assert signal_host.device.type == 'cpu' and signal_host.dtype == torch.float32 and signal_host.is_contiguous()
        N, L = signal_host.shape
        T = L // 5
        if seq_host is None:
            seq_host = torch.empty(N, T, dtype=torch.int8).pin_memory()
        if lens_host is None:
            lens_host = torch.empty(N, dtype=torch.int32).pin_memory()
        self._check(self.lib.xb_compute_scores_host(self.h, ctypes.c_void_p(signal_host.data_ptr()), N, L,
                                                    ctypes.c_void_p(seq_host.data_ptr()),
                                                    ctypes.c_void_p(lens_host.data_ptr()), _stream(self.device)),
                    'xb_compute_scores_host')
        return seq_host, lens_host

    def gemm_selftest(self, A, B):
        A, B = A.contiguous(), B.contiguous()
        M, K = A.shape
        N = B.shape[0]
        D = torch.empty(M, N, dtype=torch.float32, device=self.device)
        self._check(self.lib.xb_gemm_selftest(self.h, _ptr(A), _ptr(B), _ptr(D), M, N, K, _stream(self.device)),
                    'xb_gemm_selftest')
        return D
