"""CRF basecalling with the reference's call surface (ub-bonito/bonito/crf/basecall.py): stitch_results
(:15-24), compute_scores (:27-82, Viterbi branch), apply_stride_to_moves (:85-93), basecall (:96-119).

compute_scores runs a host batch through the host-buffer C ABI (xb_compute_scores_submit / _wait in slot 0): pinned H2D
of the chunk batch, fused stem, five persistent LSTM layers, CRF head, posteriors, max-marginal Viterbi and left-packing
on the GPU, D2H of the packed (N, T) int8 letters and their lengths.  The Python loops of the reference (ord() per
base, per-row padding) are gone; the returned dict has the same keys, dtypes and contents.
"""
import numpy as np
import torch

from ..multiprocessing import thread_iter
from ..util import chunk, stitch, batchify, unbatchify


def stitch_results(results, length, size, overlap, stride, reverse=False):
    """Stitch results together with a given overlap."""
    if isinstance(results, dict):
        return {k: stitch_results(v, length, size, overlap, stride, reverse=reverse) for k, v in results.items()}
    return stitch(results, size, overlap, length, stride, reverse=reverse)


def _pinned(model, name, shape, dtype):
    cache = model.__dict__.setdefault('_xb_pinned', {})
    buf = cache.get(name)
    if buf is None or buf.dtype != dtype or buf.numel() < int(np.prod(shape)):
        buf = torch.empty(int(np.prod(shape)), dtype=dtype).pin_memory()
        cache[name] = buf
    return buf[:int(np.prod(shape))].view(*shape)


def compute_scores(model, batch, beam_width=32, beam_cut=100.0, scale=1.0, offset=0.0, blank_score=2.0, reverse=False):
    """Compute scores for model: batch (N, 1, chunksize) host tensor -> {'sequence', 'qstring', 'moves'}."""
    head = model.encoder[-1]
    device = next(model.parameters()).device
    if device.type == 'cuda':
        torch.cuda.set_device(device)       # basecall() runs this on a pipeline thread; the current device is per-thread state
    N, _, L = batch.shape
    T = L // model.stride
    if not head.expand_blanks:
        # the reference's beam-search branch (crf/basecall.py:33-46; koi's decoder is ACGT-only, this one takes any alphabet):
        # scores without blank columns -> blank score inserted (nn.py:122-129) -> xb_crf_beam_search
        with torch.no_grad():
            scores = model(batch.to(device)).float()
        n = head.n_base
        scores = torch.nn.functional.pad(scores.view(T, N, -1, n), (1, 0, 0, 0, 0, 0, 0, 0), value=blank_score).view(T, N, -1)
        if reverse:
            scores = model.seqdist.reverse_complement(scores)
        seq, qs, moves, _ = model.seqdist.beam_search(scores, beam_width=beam_width, beam_cut=beam_cut)
        return {'qstring': qs.cpu(), 'sequence': seq.cpu(), 'moves': moves.cpu().numpy()}
    if not reverse and batch.device.type == 'cpu':
        return _collect_scores(*_submit_scores(model, batch, 0))
    # reverse complement permutes the score tensor between encoder and decode: two device calls
    with torch.no_grad():
        scores = model(batch.to(device))
    if reverse:
        scores = model.seqdist.reverse_complement(scores)
    seq, qs, lens = model.seqdist.decode_packed(scores)
    return {
        'qstring': qs.cpu(),
        'sequence': seq.cpu(),
        'moves': np.zeros((N, T), dtype=bool),
    }


def _submit_scores(model, batch, slot):
    """Host-buffer half of compute_scores: stage the batch in the slot's pinned buffer and enqueue it."""
    if not model.encoder[-1].expand_blanks or model.encoder._stem() is None:
        raise RuntimeError('the host-buffer path needs the sup@v3.3 encoder layout with expand_blanks')
    device = next(model.parameters()).device
    if device.type == 'cuda':
        torch.cuda.set_device(device)
    N, _, L = batch.shape
    T = L // model.stride
    h = model.seqdist.engine.get(device, N, T, bf16=next(model.parameters()).dtype == torch.bfloat16)
    model.encoder.sync_weights(h)
    staged = _pinned(model, 'signal%d' % slot, (N, L), torch.float32)
    staged.copy_(batch[:, 0, :])
    seq_pin, lens_pin = _pinned(model, 'seq%d' % slot, (N, T), torch.int8), _pinned(model, 'lens%d' % slot, (N,), torch.int32)
    h.compute_scores_submit(slot, staged, seq_pin, lens_pin)
    return h, slot, seq_pin, N, T


def _collect_scores(h, slot, seq_pin, N, T):
    h.compute_scores_wait(slot)
    sequence = seq_pin.clone()
    qstring = torch.where(sequence != 0, torch.tensor(ord('O'), dtype=torch.int8), torch.tensor(0, dtype=torch.int8))
    return {'qstring': qstring, 'sequence': sequence, 'moves': np.zeros((N, T), dtype=bool)}


def to_str(x):
    """koi.decode.to_str as used by the reference: drop zeros, bytes -> ascii."""
    x = np.asarray(x)
    return x[x != 0].astype('u1').tobytes().decode('ascii')


def apply_stride_to_moves(model, attrs):
    """Stitched per-read arrays -> the record the Writer consumes: letters and qualities as ascii strings (zeros dropped),
    and the move table spread onto sample positions (one flag per signal sample, set at the first sample of a step that
    emitted a base; all False for the UB models, whose decode carries no moves)."""
    step_moved = np.asarray(attrs['moves']).astype(bool)
    sig_move = np.zeros(step_moved.size * model.stride, dtype=bool)
    sig_move[np.flatnonzero(step_moved) * model.stride] = True
    return dict(sequence=to_str(attrs['sequence']), qstring=to_str(attrs['qstring']), sig_move=sig_move)


def basecall(model, reads, chunksize=4000, overlap=100, batchsize=32, reverse=False):
    """Basecalls a set of reads: iterator of (read, {'sequence', 'qstring', 'sig_move'}) in input order.

    Four stages, each drained by its own background thread through a depth-1 queue (thread_iter), as in the reference:
    reads -> chunk tensors keyed (read, 0, n_samples) -> exact-size batches -> compute_scores on the GPU -> regrouped per
    read, stitched, converted to strings."""

    def chunked():
        for read in reads:
            yield (read, 0, len(read.signal)), chunk(torch.from_numpy(read.signal), chunksize, overlap)

    def scored(batches):
        # one batch ahead on the GPU: batch i+1 is submitted (xb_compute_scores_submit: H2D, encoder, decode, D2H on their own
        # streams) before the results of batch i are collected, so the copies hide under the kernels
        in_flight = None
        for i, (keys, batch) in enumerate(batches):
            if reverse or batch.device.type != 'cpu':
                if in_flight is not None:
                    yield in_flight[0], _collect_scores(*in_flight[1:])
                    in_flight = None
                yield keys, compute_scores(model, batch, reverse=reverse)
                continue
            job = (keys,) + _submit_scores(model, batch, i & 1)
            if in_flight is not None:
                yield in_flight[0], _collect_scores(*in_flight[1:])
            in_flight = job
        if in_flight is not None:
            yield in_flight[0], _collect_scores(*in_flight[1:])

    def stitched(per_read):
        for (read, start, end), parts in per_read:
            yield read, stitch_results(parts, end - start, chunksize, overlap, model.stride, reverse)

    def finished(results):
        for read, attrs in results:
            yield read, apply_stride_to_moves(model, attrs)

    batches = thread_iter(batchify(thread_iter(chunked()), batchsize=batchsize))
    per_read = unbatchify(thread_iter(scored(batches)))
    return thread_iter(finished(thread_iter(stitched(per_read))))
