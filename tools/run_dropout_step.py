"""Cost of dropout in the training step: Trainer.train_one_step (bonito/training.py:91-117) on the sup@v3.3 UB X encoder built
with rnn_encoder(drop_rate_bottom=...) -- batch 512 x 4000 samples (T = 800), targets as in tools/run_config5.py -- with the
seven Dropout modules at p = 0 (the step launches exactly the kernels of the plain step) and at p = 0.1, alternated step by
step in one process on one model.

Reports, per arm: the step time (CUDA events around one train_one_step, median of the repeats); from a separate
torch.profiler pass, the device time per step of the kernels the masks add (dropout16_kernel: the elementwise masks of
sites 2-6; the masked transpose16v_kernel: the transposed dropped LSTM inputs of the backward) and of the kernels that take
a masked form (conv12_im2col_kernel, conv2_bwd_kernel); the extra device workspace (the one buffer the LSTM sites need);
the card's name and power limit, read in the same run.
    python tools/run_dropout_step.py [--out FILE] [--repeats R] [--N N] [--p P]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import bonito_oracle as bo                    # noqa: E402  weight generator only
from xna_basecaller_b200 import util                      # noqa: E402
from xna_basecaller_b200.training import Trainer          # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {'torch_name': torch.cuda.get_device_name(), 'nvidia_smi': q.stdout.strip() or q.stderr.strip()}


def kernel_group(name):
    if 'dropout16_kernel' in name:
        return 'dropout16_kernel (sites 2-6, elementwise)'
    if 'transpose16v_kernel' in name and ('<false, false, true>' in name or 'ILb0ELb0ELb1E' in name):
        return 'transpose16v_kernel, masked (sites 3-6, backward)'
    if 'conv12_im2col_kernel' in name:
        return 'conv12_im2col_kernel (x2: forward + backward recompute)'
    if 'conv2_bwd_kernel' in name:
        return 'conv2_bwd_kernel'
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r04_dropout_train_step.json'))
    ap.add_argument('--repeats', type=int, default=10)
    ap.add_argument('--N', type=int, default=512)
    ap.add_argument('--p', type=float, default=0.1)
    args = ap.parse_args()
    N, L = args.N, 4000
    cfg = {'global_norm': {'state_len': 3}, 'input': {'features': 1}, 'labels': {'labels': list('NACGTX')},
           'model': {'package': 'xna_basecaller_b200.crf'},
           'encoder': {'stride': 5, 'activation': 'swish', 'features': 768, 'winlen': 19, 'scale': 5.0, 'rnn_type': 'lstm',
                       'blank_score': 2.0, 'drop_rate_bottom': args.p}}
    model = util.load_symbol(cfg, 'Model')(cfg)
    sd = bo.reference_state_dict(n_base=5, seed=25)
    with torch.no_grad():        # the plain model's weights, parameter by parameter (Dropouts shift the state_dict keys)
        for q, v in zip([q for n, q in model.named_parameters()], sd.values()):
            q.copy_(v)
    drops = [m for m in model.modules() if isinstance(m, torch.nn.Dropout) and m is not model.encoder[-1].dropout]
    assert len(drops) == 7
    trainer = Trainer(model, 'cuda')
    trainer.init_optimizer(2e-3)
    model.train()
    x = torch.randn(N, 1, L, generator=torch.Generator().manual_seed(1234)).cuda()
    rs = np.random.RandomState(3)
    lens = rs.randint(350, 451, N)
    tg = np.zeros((N, int(lens.max())), dtype=np.int64)
    for i, n in enumerate(lens):
        seq = rs.randint(1, 5, n)
        cand = np.arange(5, n - 5, 11)
        seq[cand[rs.rand(len(cand)) < 0.99]] = 5
        tg[i, :n] = seq
    tg, tl = torch.from_numpy(tg).cuda(), torch.from_numpy(lens).cuda()
    torch.manual_seed(0)

    def set_p(p):
        for m in drops:
            m.p = p

    def step(p):
        set_p(p)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        losses, _ = trainer.train_one_step((x, tg, tl))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), losses['loss']

    arms = (0.0, args.p)
    for _ in range(2):
        step(0.0)
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(2):
        step(args.p)
    free1 = torch.cuda.mem_get_info()[0]
    launches = {}
    for p in arms:
        h = model.seqdist.engine.handle
        n0 = h.launches
        step(p)
        launches[p] = h.launches - n0
    times = {p: [] for p in arms}
    loss = {p: [] for p in arms}
    for r in range(args.repeats):
        for p in (arms if r % 2 == 0 else arms[::-1]):
            ms, lo = step(p)
            times[p].append(ms)
            loss[p].append(lo)

    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for p in arms:
        step(p)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                step(p)
        acc, total = {}, 0.0
        for e in prof.events():
            if e.device_type.name != 'CUDA':
                continue
            total += e.device_time
            g = kernel_group(e.name)
            if g:
                acc[g] = acc.get(g, 0.0) + e.device_time
        kernels[p] = {'per_step_ms': {g: v / 2e3 for g, v in sorted(acc.items())}, 'all_kernels_per_step_ms': total / 2e3}

    T = L // 5
    p0, p1 = arms
    med = {p: float(np.median(times[p])) for p in arms}
    added = sum(v for g, v in kernels[p1]['per_step_ms'].items() if g.startswith(('dropout16', 'transpose16v')))
    res = {
        'what': 'Trainer.train_one_step, N=%d x %d samples (T=%d), n_base 5, rnn_encoder(drop_rate_bottom): the seven Dropout '
                'modules at p=%g and p=%g, alternated step by step on one model' % (N, L, T, p0, p1),
        'device': card(),
        'repeats': args.repeats,
        'step_ms_median': {str(p): med[p] for p in arms},
        'step_ms_all': {str(p): times[p] for p in arms},
        'step_overhead_ms': med[p1] - med[p0],
        'step_overhead_percent': 100.0 * (med[p1] - med[p0]) / med[p0],
        'kernel_launches_per_step': {str(p): launches[p] for p in arms},
        'kernels_torch_profiler': {str(p): kernels[p] for p in arms},
        'added_mask_kernels_ms_per_step': added,
        'extra_workspace_bytes_computed': T * N * 768 * 2,
        'extra_workspace_bytes_measured': int(free0 - free1),
        'loss_last': {str(p): loss[p][-1] for p in arms},
    }
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
