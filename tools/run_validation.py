"""Validation step (Trainer.validate_one_step, bonito/training.py:159-181) at training size: sup@v3.3 UB X (n_base 5),
batch 512 x 4000-sample chunks, random-init weights with bench.py's calibrated head gain (decodes of ~400 bases), targets
= the decodes mutated with a seeded ~10 % substitution / insertion / deletion rate.

Times, with CUDA events (median of the repeats): forward, loss, decode, alignment (the xb_align_counts call: its copy of
the lengths to the host, then the kernel), and the whole validate_one_step; the alignment kernel on its own from a
torch.profiler pass; alignment cells per second = sum len(seq) * len(ref) / kernel time.  For scale, the plain-C checker
(oracle/c/align_exact.c, full matrices + traceback -- a stand-in, not parasail) on all host threads for the same pairs.
    python tools/run_validation.py [--out FILE] [--repeats R]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ALPHABET, CHUNK, calibrated_weights      # noqa: E402
from oracle import bonito_oracle as bo                    # noqa: E402  weight generator only
from oracle import align_exact                            # noqa: E402
from xna_basecaller_b200 import _lib, util                # noqa: E402
from xna_basecaller_b200.training import Trainer          # noqa: E402


def mutate(rs, s, rate):
    out = []
    for ch in s:
        u = rs.rand()
        if u < rate / 3:
            out.append('ACGTX'[rs.randint(5)])
        elif u < 2 * rate / 3:
            out.append(ch)
            out.append('ACGTX'[rs.randint(5)])
        elif u >= rate:
            out.append(ch)
    return ''.join(out)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {'torch_name': torch.cuda.get_device_name(), 'nvidia_smi': q.stdout.strip() or q.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r03_validation_step.json'))
    ap.add_argument('--repeats', type=int, default=20)
    ap.add_argument('--N', type=int, default=512)
    args = ap.parse_args()
    N, L = args.N, CHUNK
    dev = torch.device('cuda', 0)
    h = _lib.Handle(ALPHABET, 3, max_N=N, max_T=L // 5, device=dev)
    x = torch.randn(N, 1, L, generator=torch.Generator().manual_seed(1234)).to(dev)
    sd, gain, _ = calibrated_weights(h, bo, x[:, 0])
    h.close()
    cfg = {'global_norm': {'state_len': 3}, 'input': {'features': 1}, 'labels': {'labels': ALPHABET},
           'model': {'package': 'xna_basecaller_b200.crf'},
           'encoder': {'stride': 5, 'activation': 'swish', 'features': 768, 'winlen': 19, 'scale': 5.0, 'rnn_type': 'lstm',
                       'blank_score': 2.0}}
    model = util.load_symbol(cfg, 'Model')(cfg)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    with torch.no_grad():
        decodes = model.decode_batch(model(x).float())
    rs = np.random.RandomState(7)
    refs = [mutate(rs, d, 0.1) or 'A' for d in decodes]
    tg = np.zeros((N, max(map(len, refs))), dtype=np.int64)
    for i, r in enumerate(refs):
        tg[i, :len(r)] = [ALPHABET.index(c) for c in r]
    tg = torch.from_numpy(tg).to(dev)
    tl = torch.tensor([len(r) for r in refs], dtype=torch.int64, device=dev)
    trainer = Trainer(model, dev)

    # the parts of validate_one_step, each between CUDA events
    def parts():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        with torch.no_grad():
            ev[0].record()
            scores = model(x).float()
            ev[1].record()
            trainer.criterion(scores, tg, tl).item()
            ev[2].record()
            seq, _, seq_len = model.seqdist.decode_packed(scores)
            ev[3].record()
            counts = _lib.align_counts(seq, seq_len, ref_rows, ref_len)
            ev[4].record()
        torch.cuda.synchronize()
        return [ev[k].elapsed_time(ev[k + 1]) for k in range(4)], seq, seq_len, counts

    letters = torch.tensor(list(''.join(ALPHABET).encode()), dtype=torch.uint8, device=dev)
    ref_rows = letters[tg].view(torch.int8)
    ref_len = tl.to(torch.int32)

    def whole():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        out = trainer.validate_one_step((x, tg, tl))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3, out

    for _ in range(3):
        parts()
        whole()
    part_ms = np.array([parts()[0] for _ in range(args.repeats)])
    whole_ms = np.array([whole()[:2] for _ in range(args.repeats)])
    _, seq, seq_len, counts = parts()
    _, _, (seqs, refs_out, accs, loss) = whole()

    # the kernel alone (a separate, profiled pass)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.repeats):
            _lib.align_counts(seq, seq_len, ref_rows, ref_len)
        torch.cuda.synchronize()
    kern = [e for e in prof.events() if 'align_counts_kernel' in e.name and e.device_type.name == 'CUDA']
    kernel_ms = float(np.median([e.device_time for e in kern])) / 1e3 if kern else float('nan')

    lens_s = np.array([len(s) for s in seqs], dtype=np.int64)
    lens_r = np.array([len(r) for r in refs_out], dtype=np.int64)
    cells = int((lens_s * lens_r).sum())
    s_np, sl_np = seq.cpu().numpy(), seq_len.cpu().numpy()
    r_np, rl_np = ref_rows.cpu().numpy(), ref_len.cpu().numpy()
    threads = os.cpu_count()
    t0 = time.perf_counter()
    want = align_exact.align_counts(s_np, sl_np, r_np, rl_np, threads=threads)
    host_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(want, counts.cpu().numpy()), 'kernel counts differ from the C checker'

    med = np.median(part_ms, axis=0)
    res = {
        'what': 'Trainer.validate_one_step, N=%d x %d samples, n_base 5, head gain %.3f, targets = decodes with ~10%% '
                'seeded substitutions / insertions / deletions' % (N, L, gain),
        'device': card(),
        'repeats': args.repeats,
        'forward_ms': float(med[0]), 'loss_ms': float(med[1]), 'decode_ms': float(med[2]),
        'alignment_call_ms': float(med[3]),
        'alignment_kernel_ms': kernel_ms,
        'validate_one_step_ms_device': float(np.median(whole_ms[:, 0])),
        'validate_one_step_ms_host_wall': float(np.median(whole_ms[:, 1])),
        'alignment_cells': cells,
        'alignment_gcells_per_s': cells / (kernel_ms * 1e-3) / 1e9,
        'mean_len_seq': float(lens_s.mean()), 'mean_len_ref': float(lens_r.mean()),
        'loss': loss, 'accuracy_mean': float(np.mean(accs)), 'accuracy_median': float(np.median(accs)),
        'host_c_checker_ms': host_ms, 'host_c_checker_threads': threads,
        'host_c_checker_note': 'oracle/c/align_exact.c (full H/D/I matrices + traceback), a plain-C stand-in, not parasail',
        'kernel_equals_checker': True,
    }
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
