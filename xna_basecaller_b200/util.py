"""Host-side helpers of the basecalling path, with the reference's names and argument meaning
(ub-bonito/bonito/util.py): chunk (:152-166), stitch (:169-188), batchify / unbatchify (:191-225),
concat / select_range / size (:66-102), half_supported (:105-112), load_symbol (:228-239),
match_names (:242-258), load_model (:261-366), decode_ref and accuracy (:402-424).

These are bookkeeping over host arrays (rows a-1, a-2, a-11 of SURVEY.md section 8); the arithmetic of the
path runs in libxna_b200.so.  The read-sharded GPU pipeline (xna_basecaller_b200.pipeline) does the same
chunking and stitching on the device for whole read sets.
"""
import os
import re
from collections import OrderedDict
from glob import glob
from importlib import import_module
from itertools import groupby

import numpy as np
import torch

__dir__ = os.path.dirname(os.path.realpath(__file__))
__models__ = os.path.join(__dir__, 'models')


def _load_toml(path):
    try:
        import toml
        return toml.load(path)
    except ImportError:
        import tomllib
        with open(path, 'rb') as f:
            return tomllib.load(f)


def concat(xs, dim=0):
    """Type-agnostic concatenation (tensors, arrays, lists, strings, dicts of those)."""
    head = xs[0]
    if isinstance(head, torch.Tensor):
        return torch.cat(list(xs), dim=dim)
    if isinstance(head, np.ndarray):
        return np.concatenate(list(xs), axis=dim)
    if isinstance(head, list):
        out = []
        for x in xs:
            out.extend(x)
        return out
    if isinstance(head, str):
        return ''.join(xs)
    if isinstance(head, dict):
        return {k: concat([x[k] for x in xs], dim) for k in head}
    raise TypeError('cannot concatenate %r' % type(head))


def select_range(x, start, end, dim=0):
    """Type-agnostic x[start:end] along dim."""
    if isinstance(x, dict):
        return {k: select_range(v, start, end, dim) for k, v in x.items()}
    if dim == 0 or isinstance(x, list):
        return x[start:end]
    index = [slice(None)] * dim + [slice(start, end)]
    return x[tuple(index)]


def size(x, dim=0):
    """Type-agnostic length along dim."""
    if hasattr(x, 'shape'):
        return x.shape[dim]
    if dim == 0:
        return len(x)
    raise TypeError('%r has no dimension %d' % (type(x), dim))


def half_supported():
    """True when the current CUDA device computes in 16-bit (capability >= 7); the B200 path always does."""
    try:
        return torch.cuda.get_device_capability()[0] >= 7
    except Exception:
        return False


def chunk_starts(length, chunksize, overlap):
    """Start offsets of the chunks util.chunk cuts from a read of `length` samples (length >= chunksize).
    The first entry is 0 when a leading stub chunk is needed."""
    step = chunksize - overlap
    stub = (length - overlap) % step
    starts = list(range(stub, length - chunksize + 1, step))
    if stub > 0:
        starts.insert(0, 0)
    return starts


def chunk(signal, chunksize, overlap):
    """Overlapping windows of one read: (len,) -> (n_chunks, 1, chunksize).  Short reads are left-padded
    with zeros; a leading stub chunk covers the remainder that does not fill a whole step."""
    T = signal.shape[0]
    if chunksize == 0:
        chunks = signal[None, :]
    elif T < chunksize:
        pad = signal.new_zeros(chunksize - T)
        chunks = torch.cat([pad, signal])[None, :]
    else:
        starts = chunk_starts(T, chunksize, overlap)
        chunks = torch.stack([signal[s:s + chunksize] for s in starts])
    return chunks.unsqueeze(1)


def stitch_bounds(n_chunks, chunksize, overlap, length, stride):
    """(lo, hi) row-position slice kept from every chunk by stitch (forward direction); hi None = to the end."""
    if n_chunks == 1:
        return [(0, None)]
    semi = overlap // 2
    start, end = semi // stride, (chunksize - semi) // stride
    stub = (length - overlap) % (chunksize - overlap)
    first_end = (stub + semi) // stride if stub > 0 else end
    return [(0, first_end)] + [(start, end)] * (n_chunks - 2) + [(start, None)]


def stitch(chunks, chunksize, overlap, length, stride, reverse=False):
    """Join the per-chunk rows of one read, trimming half an overlap from each side of every seam."""
    n = chunks.shape[0]
    if n == 1:
        return chunks.squeeze(0)
    bounds = stitch_bounds(n, chunksize, overlap, length, stride)
    if not reverse:
        return concat([chunks[i][lo:hi] for i, (lo, hi) in enumerate(bounds)])
    # reversed reads: mirror every slice and walk the chunks backwards
    semi = overlap // 2
    start, end = semi // stride, (chunksize - semi) // stride
    first_end = bounds[0][1]
    rows = list(chunks)
    parts = [rows[-1][:-start]]
    parts += [x[-end:-start] for x in reversed(rows[1:-1])]
    parts.append(rows[0][-first_end:])
    return concat(parts)


def batchify(items, batchsize, dim=0):
    """Pack (key, value) items into exact `batchsize` batches; every batch carries the list of
    (key, (row_start, row_end)) spans it holds so that unbatchify can undo it."""
    held, fill = [], 0
    for key, value in items:
        n, off = size(value, dim), 0
        while off < n:
            take = min(batchsize - fill, n - off)
            held.append(((key, (fill, fill + take)), select_range(value, off, off + take, dim)))
            fill += take
            off += take
            if fill == batchsize:
                yield tuple(k for k, _ in held), concat([v for _, v in held], dim)
                held, fill = [], 0
    if held:
        yield tuple(k for k, _ in held), concat([v for _, v in held], dim)


def unbatchify(batches, dim=0):
    """Inverse of batchify: regroup consecutive spans with the same key."""
    def spans():
        for keys, value in batches:
            for key, (lo, hi) in keys:
                yield key, select_range(value, lo, hi, dim)
    for key, group in groupby(spans(), key=lambda kv: kv[0]):
        yield key, concat([v for _, v in group], dim)


def load_symbol(config, symbol):
    """Import `symbol` from the package a model's config.toml names under [model] package."""
    if not isinstance(config, dict):
        dirname = config
        if not os.path.isdir(dirname) and os.path.isdir(os.path.join(__models__, dirname)):
            dirname = os.path.join(__models__, dirname)
        config = _load_toml(os.path.join(dirname, 'config.toml'))
    return getattr(import_module(config['model']['package']), symbol)


def match_names(state_dict, model, skip_layers=()):
    """Key remap from a checkpoint to `model` by sorted tensor shape (checkpoints saved under other
    module names load as long as the shape multiset matches)."""
    def keys_and_shapes(sd):
        rows = sorted((tuple(v.shape), i, k) for i, (k, v) in enumerate(sd.items()))
        rows = [(k, s) for s, i, k in rows if k not in skip_layers]
        return [k for k, _ in rows], [s for _, s in rows]
    k1, s1 = keys_and_shapes(state_dict)
    k2, s2 = keys_and_shapes(model.state_dict())
    assert s1 == s2, 'checkpoint and model tensor shapes differ'
    remap = dict(zip(k1, k2))
    return OrderedDict((k, remap[k]) for k in state_dict if k not in skip_layers)


def load_model(dirname, device, weights=None, half=None, chunksize=None, batchsize=None, overlap=None,
               quantize=False, use_koi=False, skip_top=False, drop_rate=None, drop_rate_bottom=None):
    """Build Model from <dirname>/config.toml and load weights_<n>.tar (latest when weights is None):
    the same directory layout, overrides and key remapping as the reference loader (bonito/util.py:261-366).
    Flags override the config with the reference's `value or config` rule for chunksize / batchsize (0 falls back
    to the config) and `is not None` for overlap / drop rates.  `quantize` / `use_koi` are accepted and ignored (koi
    is bypassed for UB alphabets, bonito/util.py:299-301)."""
    if not os.path.isdir(dirname) and os.path.isdir(os.path.join(__models__, dirname)):
        dirname = os.path.join(__models__, dirname)
    if not weights:
        found = glob(os.path.join(dirname, 'weights_*.tar'))
        if not found:
            raise FileNotFoundError('no model weights found in %r' % dirname)
        weights = max(int(re.sub(r'.*_([0-9]+)\.tar', r'\1', w)) for w in found)
    config = _load_toml(os.path.join(dirname, 'config.toml'))
    bc = config.setdefault('basecaller', {})
    bc['chunksize'] = chunksize or bc.get('chunksize', 4000)
    bc['overlap'] = overlap if overlap is not None else bc.get('overlap', 500)
    bc['batchsize'] = batchsize or bc.get('batchsize', 64)
    enc = config.setdefault('encoder', {})
    enc['drop_rate'] = drop_rate if drop_rate is not None else enc.get('drop_rate', 0)
    enc['drop_rate_bottom'] = drop_rate_bottom if drop_rate_bottom is not None else enc.get('drop_rate_bottom', 0)
    Model = load_symbol(config, 'Model')
    model = Model(config)
    path = os.path.join(dirname, 'weights_%s.tar' % weights)
    state = torch.load(path, map_location='cpu')
    state = {k.replace('module.', ''): v for k, v in state.items()}
    skip = [k for k in model.state_dict() if k.startswith('encoder.9')] if skip_top else []
    names = match_names(state, model, skip)
    result = model.load_state_dict(OrderedDict((names[k], v) for k, v in state.items() if k in names),
                                   strict=not skip_top)
    assert list(result.unexpected_keys) == [], 'checkpoint holds tensors the model does not: %s' % result.unexpected_keys
    assert list(result.missing_keys) == skip, 'model tensors missing from the checkpoint: %s' % result.missing_keys
    if half is None:
        half = half_supported()
    if half:
        model = model.half()
    model.eval()
    model.to(device)
    return model


def decode_ref(encoded, labels):
    """The letters of the non-zero (1-based) labels of one target row."""
    return ''.join(labels[e] for e in encoded.tolist() if e)


def _accuracy(counts, ref_len, balanced, min_coverage):
    """The reference's accuracy expressions on one pair's (score, eq, x, ins, del), in Python float arithmetic.  The
    coverage of the reference counts the alignment's columns, gaps included.  An empty alignment, or an empty reference,
    scores 0 (the reference would divide by zero)."""
    _, eq, x, ins, dl = (int(c) for c in counts)
    r_coverage = (eq + x + ins + dl) / ref_len if ref_len else 0.0
    if r_coverage < min_coverage:
        return 0.0
    if balanced:
        den = eq + x + dl
        return (eq - ins) / den * 100 if den else 0.0
    den = eq + ins + x + dl
    return eq / den * 100 if den else 0.0


def accuracy_batch(seq, seq_len, ref, ref_len, balanced=False, min_coverage=0.0):
    """accuracy() of every row pair of device tensors: seq / ref (N, *) int8 left-packed letter rows, lengths (N,).
    The alignments run in one xb_align_counts call; only the (N, 5) counts come back.  Returns a list of N floats."""
    from ._lib import align_counts
    counts = align_counts(seq, seq_len, ref, ref_len).cpu().tolist()
    ref_lens = ref_len.cpu().tolist()
    return [_accuracy(c, rl, balanced, min_coverage) for c, rl in zip(counts, ref_lens)]


def accuracy(ref, seq, balanced=False, min_coverage=0.0):
    """Percent identity of the best local alignment of `seq` against `ref` (host strings), computed on the current CUDA
    device: 100 * '=' / ('=' + 'I' + 'X' + 'D'), or with balanced 100 * ('=' - 'I') / ('=' + 'X' + 'D'); 0 when the
    alignment covers less than min_coverage of ref.  Scoring and tie rules: csrc/align.cu."""
    dev = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else None
    if dev is None:
        raise RuntimeError('xna_basecaller_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    s, r = seq.encode(), ref.encode()
    rows = torch.zeros(2, max(len(s), len(r), 1), dtype=torch.uint8)
    rows[0, :len(s)] = torch.frombuffer(bytearray(s), dtype=torch.uint8) if s else rows[0, :0]
    rows[1, :len(r)] = torch.frombuffer(bytearray(r), dtype=torch.uint8) if r else rows[1, :0]
    rows = rows.view(torch.int8).to(dev)
    lens = torch.tensor([[len(s)], [len(r)]], dtype=torch.int32, device=dev)
    return accuracy_batch(rows[:1], lens[0], rows[1:], lens[1], balanced, min_coverage)[0]
