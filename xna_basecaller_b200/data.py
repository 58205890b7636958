"""Training data path (SURVEY 8f N3): the reference's numpy chunk datasets (ub-bonito/bonito/data.py) for the training step
of this package.

What is mirrored, with the reference's names and return values:
  load_numpy_datasets(limit, directory, load_bkps)   data.py:129-163   chunks.npy / references.npy / reference_lengths.npy,
                                                                       optional indices.npy sub-sampling, `limit`
  load_numpy(limit, directory, ...)                   data.py:100-126   train / validation split (validation/ directory, else
                                                                       97 % / 3 %), DataLoader keyword dictionaries
  ChunkDataSet                                        data.py:10-87     (chunk (1, L) float32, target int64, length int64) items

What is new: DeviceChunkLoader.  The reference feeds the GPU through a torch DataLoader with up to 32 worker processes
(README.md:116); a B200 has room for the whole data set (10^6 chunks of 4000 fp16 samples are 8 GB of its 180 GB), so the
chunks, targets and lengths are uploaded ONCE and every batch is an index gather on the device -- shuffling is a device
permutation, there are no workers, no pinned staging and no per-step host-to-device copy.  It yields the (data, targets,
lengths) batches Trainer.train_one_step consumes and has the `len()` / `.sampler` surface the reference's epoch loop reads.

Not built: the on-the-fly spliced / spiked unnatural-base augmentation (stitch_chunks.py:323-454, spike_chunks.py:247-297:
numpy procedures over pandas k-mer tables, driven by one numpy Generator stream per data set item; DESIGN.md section 7).
Passing spike_kwargs / stitch_kwargs raises NotImplementedError instead of silently training on un-augmented data.  (The
model-side regulariser of the same training setup, rnn_encoder's drop_rate_bottom dropout, is built: training.py.)
"""
import os

import numpy as np
import torch


def _no_augmentation(spike_kwargs, stitch_kwargs):
    if spike_kwargs is not None or stitch_kwargs is not None:
        raise NotImplementedError('the spliced / spiked UB augmentation (bonito/stitch_chunks.py, spike_chunks.py) is not part of '
                                  'this package: prepare augmented chunks with the reference and load them as plain .npy sets')


class ChunkDataSet:
    """Items of a chunk data set as the reference returns them: chunk (1, L) float32, target int64, length int64."""

    def __init__(self, chunks, targets, lengths, breakpoints=None, spike_kwargs=None, stitch_kwargs=None, epoch_reset_seed=False):
        _no_augmentation(spike_kwargs, stitch_kwargs)
        self.chunks = np.expand_dims(chunks, axis=1)
        self.targets = targets
        self.lengths = lengths
        self.breakpoints = breakpoints
        self.replace_6_letter = False      # data.py:82-83: Y -> X for five-letter models

    def __getitem__(self, i):
        chunk = self.chunks[i].astype(np.float32)
        target = self.targets[i].astype(np.int64)
        length = self.lengths[i].astype(np.int64)
        if self.replace_6_letter:
            target[target == 6] = 5
        return chunk, target, length

    def __len__(self):
        return len(self.lengths)


def load_numpy_datasets(limit=None, directory=None, load_bkps=False):
    """chunks, targets, lengths (and breakpoints with load_bkps) of a ctc-data directory."""
    path = lambda name: os.path.join(directory, name)
    chunks = np.load(path('chunks.npy'), mmap_mode='r')
    targets = np.load(path('references.npy'), mmap_mode='r')
    lengths = np.load(path('reference_lengths.npy'), mmap_mode='r')
    if os.path.exists(path('indices.npy')):
        idx = np.load(path('indices.npy'), mmap_mode='r')
        idx = idx[idx < lengths.shape[0]]
        if limit:
            idx = idx[:limit]
        out = [chunks[idx, :], targets[idx, :], lengths[idx]]
        if load_bkps:
            out.append(np.load(path('breakpoints.npy'), mmap_mode='r')[idx, :])
        return tuple(out)
    n = limit if limit else lengths.shape[0]
    out = [np.array(chunks[:n]), np.array(targets[:n]), np.array(lengths[:n])]
    if load_bkps:
        out.append(np.array(np.load(path('breakpoints.npy'), mmap_mode='r')[:n]))
    return tuple(out)


def load_numpy(limit, directory, spike_kwargs=None, stitch_kwargs=None):
    """(train_loader_kwargs, valid_loader_kwargs) for the data in `directory`: keyword dictionaries for a DataLoader --
    or for DeviceChunkLoader, which takes the same `dataset` / `shuffle` keys."""
    _no_augmentation(spike_kwargs, stitch_kwargs)
    train = load_numpy_datasets(limit=limit, directory=directory)
    vdir = os.path.join(directory, 'validation')
    if os.path.exists(vdir):
        valid = load_numpy_datasets(directory=vdir)
    else:
        print('[validation set not found: splitting training set (97%-3%)]')
        split = int(np.floor(len(train[0]) * 0.97))
        valid = [x[split:] for x in train]
        train = [x[:split] for x in train]
    return ({'dataset': ChunkDataSet(*train), 'shuffle': True},
            {'dataset': ChunkDataSet(*valid, epoch_reset_seed=True), 'shuffle': False})


class _Sampler:
    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n


class DeviceChunkLoader:
    """Batches of a ChunkDataSet served from device memory (see the module docstring).

    dataset: ChunkDataSet (or anything with .chunks (n, 1, L), .targets (n, Lmax), .lengths (n)).
    Iterating yields (data (B, 1, L) float32, targets (B, Lmax) int64, lengths (B,) int64) on `device`; one pass covers every
    item once (the last batch may be short, as with DataLoader's drop_last=False).  With shuffle the order is a fresh device
    permutation per pass from a generator seeded with `seed`, so runs are reproducible.
    batch_multiple: the training step of this package needs batches that are multiples of 8 (TMA alignment, train_bwd.cu);
    with batch_multiple=8 the last batch of a pass is cut down to a multiple of 8 and the left-over (< 8) items wait for
    the next pass's permutation."""

    def __init__(self, dataset, batch_size=512, shuffle=False, device='cuda', seed=0, storage_dtype=torch.float16,
                 batch_multiple=1, **_unused):
        self.device = torch.device(device)
        self.batch_size, self.shuffle, self.batch_multiple = int(batch_size), bool(shuffle), int(batch_multiple)
        if self.batch_size % self.batch_multiple:
            raise ValueError('batch_size must be a multiple of batch_multiple')
        chunks = np.asarray(dataset.chunks)
        if chunks.ndim == 3:
            chunks = chunks[:, 0, :]
        # fp16 in HBM (the training forward reads fp16 operands anyway; the reference's chunks.npy are float16 files)
        self.chunks = torch.from_numpy(np.ascontiguousarray(chunks)).to(self.device, storage_dtype)
        self.targets = torch.from_numpy(np.ascontiguousarray(dataset.targets).astype(np.int64)).to(self.device)
        self.lengths = torch.from_numpy(np.ascontiguousarray(dataset.lengths).astype(np.int64)).to(self.device)
        if getattr(dataset, 'replace_6_letter', False):
            self.targets[self.targets == 6] = 5
        self.sampler = _Sampler(len(self.lengths))
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(seed)

    def __len__(self):
        n = len(self.lengths) - len(self.lengths) % self.batch_multiple
        return (n + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        n = len(self.lengths)
        order = torch.randperm(n, device=self.device, generator=self._gen) if self.shuffle else torch.arange(n, device=self.device)
        n_used = n - n % self.batch_multiple
        for lo in range(0, n_used, self.batch_size):
            idx = order[lo:min(lo + self.batch_size, n_used)]
            yield (self.chunks.index_select(0, idx).unsqueeze(1).float(), self.targets.index_select(0, idx),
                   self.lengths.index_select(0, idx))
