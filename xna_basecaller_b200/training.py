"""The training step with the reference's Trainer surface (ub-bonito/bonito/training.py:71-117, 183-187).

train_one_step = zero_grad -> scores = model(data) -> loss = criterion(scores, targets, lengths) -> backward -> gradient-norm
clip at 2.0 -> AdamW step.  Here the forward / loss / backward run through libxna_b200.so (xb_encoder_fwd_train,
xb_ctc_crf_loss_fwd / _bwd, xb_encoder_bwd behind torch.autograd.Function nodes) and the clip + AdamW update is one fused
multi-tensor call (xb_adamw_step).  Gradients are transported as bf16 with fp32 accumulation, so there is no GradScaler
(`use_amp` is accepted for signature compatibility and ignored).  Data loading / augmentation stay with the caller.

Models built with rnn_encoder(drop_rate_bottom=p) train with their dropout: the fused step applies it on the GPU
(xb_encoder_fwd_train_dropout) with masks drawn from one seed per forward that Serial.forward takes from torch's default
CPU generator, so torch.manual_seed makes a run repeatable.  Not built: the head's dropout (LinearCRFEncoder(drop_rate > 0)
raises in training: where the reference applies it in the head's forward is not recorded here) and the spliced / spiked
augmentation (see data.py).

validate_one_step / validate_one_epoch (training.py:159-181) score the validation chunks on the device: forward, loss,
one CRF decode, and the local alignment of every decode against its reference (xb_align_counts) -- only the strings,
the loss and 20 bytes of alignment counts per chunk come back to the host.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .util import _accuracy
from .schedule import linear_warmup_cosine_decay


class AdamW(torch.optim.Optimizer):
    """torch.optim.AdamW's state layout and hyper-parameters ('lr', 'betas', 'eps', 'weight_decay'; state 'step', 'exp_avg',
    'exp_avg_sq'), stepped by xb_adamw_step together with clip_grad_norm_(max_norm).  step(max_norm) returns the total
    gradient norm before clipping, like torch.nn.utils.clip_grad_norm_."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._scratch = None
        self._norm = None

    @torch.no_grad()
    def step(self, max_norm=0.0):
        lib = _lib.load()
        total = None
        for group in self.param_groups:
            ps = [p for p in group['params'] if p.grad is not None]
            if not ps:
                continue
            for p in ps:
                if p.dtype != torch.float32 or not p.is_cuda:
                    raise RuntimeError('xb_adamw_step updates fp32 CUDA parameters (master weights)')
                st = self.state[p]
                if not st:
                    st['step'] = 0
                    st['exp_avg'] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st['step'] += 1
            dev = ps[0].device
            grads = [p.grad.contiguous() for p in ps]
            n = len(ps)
            blocks = sum((p.numel() + 65535) // 65536 for p in ps)
            if self._scratch is None or self._scratch.numel() < blocks + 1 or self._scratch.device != dev:
                self._scratch = torch.empty(blocks + 1, dtype=torch.float32, device=dev)
                self._norm = torch.empty(1, dtype=torch.float32, device=dev)
            arr = lambda ts: (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])
            numel = (ctypes.c_int64 * n)(*[p.numel() for p in ps])
            b1, b2 = group['betas']
            rc = lib.xb_adamw_step(arr(ps), arr(grads), arr([self.state[p]['exp_avg'] for p in ps]),
                                   arr([self.state[p]['exp_avg_sq'] for p in ps]), numel, n, float(group['lr']), float(b1),
                                   float(b2), float(group['eps']), float(group['weight_decay']), float(max_norm),
                                   int(self.state[ps[0]]['step']), ctypes.c_void_p(self._norm.data_ptr()),
                                   ctypes.c_void_p(self._scratch.data_ptr()),
                                   ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            if rc != 0:
                raise RuntimeError('xb_adamw_step failed (%d): %s' % (rc, lib.xb_last_error(None).decode()))
            for p in ps:      # the kernel wrote through raw pointers: tell torch (and the engine's weight stamps) they changed
                torch.autograd.graph.increment_version(p)
            total = self._norm if total is None else torch.sqrt(total ** 2 + self._norm ** 2)
        return total


class Trainer:
    """Trainer.train_one_step / validate_one_step / validate_one_epoch / init_optimizer / get_lr_scheduler of the
    reference; the epoch loop and checkpoints stay in the reference's own training.py, which can drive this object
    unchanged."""

    def __init__(self, model, device, train_loader=None, valid_loader=None, criterion=None, use_amp=True,
                 lr_scheduler_fn=None, restore_optim=False, save_optim_every=10, grad_accum_split=1):
        self.model = model.to(device)
        self.device = device
        self.train_loader, self.valid_loader = train_loader, valid_loader
        self.criterion = criterion or model.seqdist.ctc_loss
        self.use_amp = use_amp
        self.lr_scheduler_fn = lr_scheduler_fn or linear_warmup_cosine_decay()
        self.restore_optim, self.save_optim_every = restore_optim, save_optim_every
        self.grad_accum_split = grad_accum_split
        self.optimizer = None

    def init_optimizer(self, lr, **kwargs):
        self.optimizer = AdamW([p for p in self.model.parameters() if p.requires_grad], lr=lr, **kwargs)

    def get_lr_scheduler(self, epochs, last_epoch=0):
        return self.lr_scheduler_fn(self.optimizer, self.train_loader, epochs, last_epoch)

    def train_one_step(self, batch):
        self.optimizer.zero_grad()
        self.model.train()
        losses = None
        for data_, targets_, lengths_ in zip(*map(lambda t: t.chunk(self.grad_accum_split, dim=0), batch)):
            data_, targets_, lengths_ = data_.to(self.device), targets_.to(self.device), lengths_.to(self.device)
            scores_ = self.model(data_)
            losses_ = self.criterion(scores_.to(torch.float32), targets_, lengths_)
            if not isinstance(losses_, dict):
                losses_ = {'loss': losses_}
            losses_['loss'] = losses_['loss'] / self.grad_accum_split
            losses_['loss'].backward()
            losses = {k: (v.item() if losses is None else v.item() + losses[k]) for k, v in losses_.items()}
        grad_norm = self.optimizer.step(max_norm=2.0).item()
        return losses, grad_norm

    def validate_one_step(self, batch):
        """(seqs, refs, accs, losses) of one validation batch: the decoded strings, the references (decode_ref of the
        targets), accuracy(ref, seq, min_coverage=0.5) per chunk (0 for an empty decode) and the loss."""
        data, targets, lengths = batch[:3]
        self.model.eval()
        with torch.no_grad():
            targets, lengths = targets.to(self.device), lengths.to(self.device)
            scores = self.model(data.to(self.device)).to(torch.float32)
            losses = self.criterion(scores, targets, lengths)
            losses = {k: v.item() for k, v in losses.items()} if isinstance(losses, dict) else losses.item()
            seq, _, seq_len = self.model.seqdist.decode_packed(scores)
            # reference rows on the device: the non-zero labels moved to the front in order, then letters gathered
            packed = targets.gather(1, torch.sort((targets == 0).to(torch.int8), dim=1, stable=True).indices)
            letters = torch.tensor(list(''.join(self.model.alphabet).encode()), dtype=torch.uint8, device=scores.device)
            ref = letters[packed].view(torch.int8)
            ref_len = (targets != 0).sum(1).to(torch.int32)
            counts = _lib.align_counts(seq, seq_len, ref, ref_len).cpu().tolist()
            seq_h, seq_len_h = seq.cpu().numpy(), seq_len.cpu().tolist()
            ref_h, ref_len_h = ref.cpu().numpy(), ref_len.cpu().tolist()
        seqs = [seq_h[i, :n].astype('u1').tobytes().decode() for i, n in enumerate(seq_len_h)]
        refs = [ref_h[i, :n].astype('u1').tobytes().decode() for i, n in enumerate(ref_len_h)]
        accs = [_accuracy(c, rl, False, 0.5) if sl else 0. for c, rl, sl in zip(counts, ref_len_h, seq_len_h)]
        return seqs, refs, accs, losses

    def validate_one_epoch(self):
        """(mean loss, mean accuracy, median accuracy) over valid_loader."""
        self.model.eval()
        with torch.no_grad():
            seqs, refs, accs, losses = zip(*(self.validate_one_step(batch) for batch in self.valid_loader))
        accs = sum(accs, [])
        loss = np.mean([(x['loss'] if isinstance(x, dict) else x) for x in losses])
        return loss, np.mean(accs), np.median(accs)
