#!/usr/bin/env python
"""bench.py -- signal samples/sec basecalled (sup@v3.3 XNA) on B200, with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dtype fp16|bf16] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: BASELINE.json configs[1] = sup@v3.3 architecture,
UB "X" alphabet (n_base 5), batch 512 x 4000-sample chunks: conv stem -> 5 LSTMs -> CRF head -> CRF
posteriors -> max-marginal Viterbi -> left-packed base strings.  Metric (bonito/cli/basecaller.py:153-161):
input signal samples consumed per second.

  value   whole-job samples/s with the batch already resident in HBM (device-timed, max over ranks)
  e2e     same metric through the host-buffer C-ABI calls xb_compute_scores_submit / _wait (the pipelined form of
          xb_compute_scores_host that crf.basecall() uses): pinned host signal in, H2D + encoder + decode + D2H of packed
          strings of every step inside the timed region, batch i+1 submitted before batch i is collected
  roofline  dominant kernel (LSTM recurrence, tensor-core bound): algorithmic FLOPs / CUDA-event time
  cpu_baseline  the oracle's restatement of the reference CPU path, timed on this box's host cores on a
          bounded sample (rank 0, N=1 only)

--impl reference times the reference's own CPU implementation of the path (its torch modules as restated
in oracle/bonito_oracle.py + the C CRF decode) on the host cores, same metric.
Multi-GPU (torchrun): each rank runs the same batch shape on its own GPU (reads/chunks shard with no
data-path collective -> weak scaling); NCCL only gathers the timing / counters.

--dump-outputs DIR writes what the last timed step returned on rank 0 (default workload): DIR/seq.npy, the (N, T)
left-packed letter codes, and DIR/lens.npy, the (N,) decoded lengths, both float32 (exact for these integers).  Signal
and weights are seeded, so two builds run with the same arguments can be compared output for output (the head gain is
calibrated from decoded lengths; --head-gain pins it).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALPHABET = ['N', 'A', 'C', 'G', 'T', 'X']
N_BASE, STATE_LEN, FEATURES = 5, 3, 768
CHUNK, BATCH = 4000, 512
T_STEPS = CHUNK // 5
FLOP_PER_CHUNK = {   # SURVEY.md 8(d), 2*MAC
    'conv': 2 * (4 * 1 * 5 * 4000 + 16 * 4 * 5 * 4000 + 768 * 16 * 19 * 800),
    'lstm': 5 * 800 * 2 * (2 * 3072 * 768),
    'head': 2 * 768 * 625 * 800,
}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return {'hbm_gbs': p['hbm_gbs'], 'tf_burst': p['bf16_tflops'], 'tf_sustained': p['bf16_tflops_sustained'],
                'source': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'tf_burst': 1590.0, 'tf_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        try:                                            # NVML: a sample every 20 ms (nvidia-smi needs ~50 ms per call)
            import pynvml
            pynvml.nvmlInit()
            dev = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(dev, pynvml.NVML_CLOCK_SM)
            bits = {'hw_slowdown': pynvml.nvmlClocksThrottleReasonHwSlowdown,
                    'hw_thermal_slowdown': pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    'sw_thermal_slowdown': pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                    'sw_power_cap': pynvml.nvmlClocksThrottleReasonSwPowerCap}
            names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
            while not self.stop_flag.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(dev, pynvml.NVML_CLOCK_SM)
                reasons = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(dev)
                watts = pynvml.nvmlDeviceGetPowerUsage(dev) / 1000.0
                self.rows.append([str(sm), str(mx), str(watts)] + ['Active' if reasons & bits[n] else 'Not Active' for n in names])
                self.stop_flag.wait(0.02)
            return
        except Exception:
            pass
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(',')])
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def dump_outputs(dirname, arrays):
    """Write each tensor as dirname/<name>.npy in float32."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), t.cpu().numpy().astype(np.float32))


def workload_config(N, L):
    return {'workload': 'configs[1]: sup@v3.3 UB X (n_base 5), batch %d x %d-sample chunks per GPU, conv stem + '
                        '5 LSTM + CRF head + posteriors + Viterbi + left-pack (fused route xb_basecall_chunks); random-init '
                        'weights with the head gain calibrated for decodes that mix blanks and moves; '
                        'per-step working set (activations 0.6 GB, gates 2.5 GB, scores 1.2 GB) exceeds the 126 MB L2, '
                        'no explicit flush' % (N, L),
            'batch_per_gpu': N, 'chunk': L, 'n_base': N_BASE, 'sharding': 'chunks across GPUs, no collective'}


def cpu_reference_pass(n_chunks, threads, sd=None, repeats=1):
    """One pass of the reference CPU path over n_chunks chunks: fp32 torch encoder (the reference's own
    modules, restated) + CRF decode (C restatement) + left-pack.  Returns seconds per pass (best)."""
    from oracle import bonito_oracle as bo
    from oracle import cexact
    torch.set_num_threads(threads)
    if sd is None:
        sd = bo.reference_state_dict(n_base=N_BASE, seed=25)
    x = torch.randn(n_chunks, 1, CHUNK, generator=torch.Generator().manual_seed(1234))
    best = float('inf')
    for _ in range(repeats):
        t0 = time.perf_counter()
        with torch.no_grad():
            scores = bo.encoder_forward(sd, x, N_BASE, library=True)
        labels = cexact.crf_decode_threads(scores.numpy(), N_BASE, threads=threads)
        cexact.pack(labels, ALPHABET)
        best = min(best, time.perf_counter() - t0)
    return best


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_chunks = 64                                     # = BASELINE.json configs[0]
    cpu_reference_pass(4, cores)                      # warm-up (thread pools, page-in)
    times = []
    for _ in range(args.warmup):
        cpu_reference_pass(n_chunks, cores)
    for _ in range(args.steps):
        times.append(cpu_reference_pass(n_chunks, cores))
    total = sum(times)
    value = n_chunks * CHUNK * len(times) / total
    line = {
        'impl': 'reference', 'metric': 'signal samples/sec basecalled (sup@v3.3 XNA)', 'value': value, 'unit': 'samples/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / len(times),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': dict(workload_config(args.batch, CHUNK), sample='each step = %d chunks of the %d-chunk batch on the '
                                                                  'host CPU' % (n_chunks, args.batch)),
        'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d chunks x %d samples per step (torch fp32 encoder + C CRF decode, both on all '
                                   '%d host threads)' % (n_chunks, CHUNK, cores)},
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def calibrated_weights(h, bo, x_dev, seed=25, gain=None):
    """Random-init weights of the sup@v3.3 architecture whose CRF head gain is calibrated so that decodes MIX blanks and
    moves (SURVEY 8d: a plain random-init head decodes every chunk to the empty string, a strongly amplified one emits a base
    at every step; either way left-packing and stitching would have nothing to do).  Returns (state_dict, gain, mean length)."""
    sd = bo.reference_state_dict(n_base=N_BASE, seed=seed)
    w0 = sd['encoder.9.linear.weight'].clone()
    if gain is not None:                             # --head-gain: skip the calibration (profiling runs)
        sd['encoder.9.linear.weight'] = w0 * gain
        h.load_weights(sd)
        return sd, gain, float('nan')
    lo, hi, best = 0.02, 8.0, None                   # decoded length grows with the gain: bisect in log space
    for _ in range(12):
        gain = (lo * hi) ** 0.5
        sd['encoder.9.linear.weight'] = w0 * gain
        h.load_weights(sd)
        _, _, lens = h.basecall_chunks(x_dev[:32])
        mean = lens.float().mean().item()
        if best is None or abs(mean - 400) < abs(best[1] - 400):
            best = (gain, mean)
        if 300 <= mean <= 500:
            break
        lo, hi = (gain, hi) if mean < 400 else (lo, gain)
    sd['encoder.9.linear.weight'] = w0 * best[0]
    h.load_weights(sd)
    return sd, best[0], best[1]


def gpu_comparator(sd, dev, N):
    """The reference's PyTorch path on THIS GPU (BASELINE.md section 4): its nn modules in fp16 through torch's cuDNN LSTM /
    cuBLAS / cuDNN convolutions (oracle/bonito_oracle.py restates the module graph functionally; weights identical), and the
    restated-seqdist torch ops for the CRF decode on a 32-chunk slice scaled to N (the real seqdist wheel is unavailable)."""
    from oracle import bonito_oracle as bo
    sdh = {k: v.to(dev).half() for k, v in sd.items()}
    x = torch.randn(N, 1, CHUNK, generator=torch.Generator().manual_seed(1234)).to(dev).half()

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps, out

    with torch.no_grad():
        enc_ms, scores = timed(lambda: bo.encoder_forward(sdh, x, N_BASE, library=True), 3)
        crf = bo.CRF(STATE_LEN, ALPHABET)
        for name in ('idx', 'src_edges', 'src_dst'):
            if hasattr(crf, name):
                setattr(crf, name, getattr(crf, name).to(dev))
        nd = min(N, 32)
        sub = scores[:, :nd].float().contiguous()
        dec_ms, _ = timed(lambda: crf.viterbi((crf.posteriors(sub, 'log') + 1e-8).log()), 1)
    dec_full = dec_ms * N / nd
    return {'what': 'reference PyTorch path on the same GPU (torch %s: cuDNN LSTM fp16 + cuBLAS encoder; restated-seqdist '
                    'torch CRF decode timed on %d chunks and scaled)' % (torch.__version__, nd),
            'encoder_ms': enc_ms, 'encoder_samples_per_s': N * CHUNK / (enc_ms / 1e3),
            'decode_ms_scaled': dec_full, 'samples_per_s': N * CHUNK / ((enc_ms + dec_full) / 1e3)}


def train_step_leg(dev, N):
    """BASELINE configs[4] ("fwd_bwd"): one CTC-CRF training step of the sup@v3.3 UB X model through the plugin classes
    (crf.Model -> Trainer.train_one_step: forward, loss, backward to all 28 parameter tensors, clip_grad_norm_(2.0), AdamW),
    batch N x 4000 samples, targets ~U(350, 450) bases with ~9 % X spliced in.  A side measurement of the default bench run
    (the headline metric is basecalling), device-timed, inputs resident in HBM."""
    import numpy as np
    from oracle import bonito_oracle as bo            # weight generator only
    from xna_basecaller_b200.crf import Model
    from xna_basecaller_b200.training import Trainer
    model = Model(sup_config())
    model.load_state_dict(bo.reference_state_dict(n_base=N_BASE, seed=25))
    trainer = Trainer(model, dev)
    trainer.init_optimizer(2e-3)
    model.train()
    x = torch.randn(N, 1, CHUNK, generator=torch.Generator().manual_seed(1234)).to(dev)
    rs = np.random.RandomState(3)
    lens = rs.randint(350, 451, N)
    tg = np.zeros((N, int(lens.max())), dtype=np.int64)
    for i, n in enumerate(lens):
        seq = rs.randint(1, 5, n)
        cand = np.arange(5, n - 5, 11)
        seq[cand[rs.rand(len(cand)) < 0.99]] = 5
        tg[i, :n] = seq
    tg, tl = torch.from_numpy(tg).to(dev), torch.from_numpy(lens).to(dev)
    for _ in range(2):
        losses, _ = trainer.train_one_step((x, tg, tl))
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        losses, _ = trainer.train_one_step((x, tg, tl))
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    out = {'config': 'configs[4]: training step (fwd + CTC-CRF loss + bwd + clip + AdamW), batch %d x %d samples, fp16 forward '
                     'operands, bf16 gradient transport, fp32 accumulation and master weights' % (N, CHUNK),
           'ms_per_step': ms, 'samples_per_s': N * CHUNK / ms * 1e3, 'loss': float(losses['loss'])}
    del trainer, model
    torch.cuda.empty_cache()
    return out


def sup_config():
    return {'global_norm': {'state_len': STATE_LEN}, 'input': {'features': 1}, 'labels': {'labels': list(ALPHABET)},
            'model': {'package': 'xna_basecaller_b200.crf'},
            'encoder': {'stride': 5, 'activation': 'swish', 'features': FEATURES, 'winlen': 19, 'scale': 5.0,
                        'rnn_type': 'lstm', 'blank_score': 2.0}}


def run_readset(args, rank, world, local):
    """BASELINE configs[3]: a synthetic read set (lengths ~ N(10 k, 1 k) clipped to [4 k, 20 k], seed 11; chunksize 4000,
    overlap 500), sharded BY READ over the GPUs of the box -- strong scaling: the read set is fixed, `value` = its samples /
    max-over-ranks time.  Reads travel in blocks of --block-reads reads:
      value  blocks assigned k mod G, every rank's reads resident in HBM before the clock starts; device-timed
             (chunk gather, fused encoder + decode, stitch, D2H of the letters)
      e2e    blocks pulled DYNAMICALLY from one shared work queue (the process group's store), every block staged from host
             memory into pinned memory, uploaded, basecalled, stitched, and its base STRINGS cut on the host -- all inside
             the timed region, the three phases of consecutive blocks overlapped (ReadSetBasecaller.basecall_stream)."""
    import numpy as np
    import torch.distributed as dist
    from oracle import bonito_oracle as bo            # weights generator only
    from xna_basecaller_b200 import pipeline
    from xna_basecaller_b200.crf import Model

    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    store = dist.distributed_c10d._get_default_store() if world > 1 else None
    n_reads, B = args.reads, args.block_reads
    lengths = np.clip(np.random.RandomState(11).normal(10000, 1000, size=n_reads), 4000, 20000).astype(np.int64)
    n_blocks = (n_reads + B - 1) // B
    pool = torch.randn(1 << 26, generator=torch.Generator().manual_seed(1234)).numpy()      # 64 Mi samples of N(0,1) signal
    starts = np.random.RandomState(12).randint(0, len(pool) - 20000, size=n_reads)

    def block(k):
        return [pool[starts[r]:starts[r] + lengths[r]] for r in range(k * B, min((k + 1) * B, n_reads))]

    model = Model(sup_config())
    caller = pipeline.ReadSetBasecaller(model.half().eval().to(dev), CHUNK, 500, args.batch)
    h = caller._handle(args.batch)
    x_cal = torch.randn(64, CHUNK, generator=torch.Generator().manual_seed(5)).to(dev)
    sd, gain, _ = calibrated_weights(h, bo, x_cal, gain=args.head_gain)
    caller.model.load_state_dict(sd)
    caller.model.half()
    caller._handle(args.batch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- value: static k mod G, reads resident in HBM
    mine = list(range(rank, n_blocks, world))
    staged = [caller.stage(block(k), slot=j & 1) for j, k in enumerate(mine)]      # uploads stay resident (device tensors kept)
    for _ in range(max(args.warmup, 1)):
        caller.finish(caller.launch(caller.stage(block(0))))
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = h.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    bases = chunks = 0
    for _ in range(args.steps):
        prev = None
        for blk in staged + [None]:                      # block i+1 is enqueued before block i's letters are collected
            cur = caller.launch(dict(blk)) if blk is not None else None
            if prev is not None:
                strings, c = caller.finish(prev)
                chunks += c['chunks']
                bases += sum(len(s) for s in strings)
            prev = cur
    e1.record()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = h.launches - launches0
    my_samples = int(sum(b['lengths'].sum() for b in staged if b['n_reads']))
    del staged

    # ---- e2e: dynamic queue, host-resident reads, strings on the host
    barrier()
    t0 = time.perf_counter()
    e2e_reads = 0
    phase = {'seconds_stage_h2d': 0.0, 'seconds_gpu_batches': 0.0, 'seconds_strings': 0.0}
    for step in range(args.steps):
        queue = pipeline.WorkQueue(n_blocks, store=store, key='xb_readset_pass_%d' % step)
        for strings, c in caller.basecall_stream(block(k) for k in queue):
            e2e_reads += c['reads']
            for k_ in phase:
                phase[k_] += c[k_]
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    clocks = sampler.summary()

    table = pipeline.gather_counters({'dev_ms': dev_ms, 'e2e_ms': e2e_s * 1e3, 'samples': my_samples, 'chunks': chunks,
                                      'bases': bases, 'e2e_reads': e2e_reads, 'launches': launches,
                                      'stage_s': phase['seconds_stage_h2d'], 'gpu_s': phase['seconds_gpu_batches'],
                                      'strings_s': phase['seconds_strings']},
                                     device=dev if world > 1 else None)
    if rank == 0:
        total = float(lengths.sum())
        dev_ms, e2e_ms = max(table['dev_ms']), max(table['e2e_ms'])
        n_chunks = sum(table['chunks']) / args.steps
        line = {
            'metric': 'signal samples/sec basecalled (sup@v3.3 XNA)', 'value': total * args.steps / (dev_ms / 1e3),
            'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 1),
            'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'fp16', 'data': 'synthetic',
            'config': {'workload': 'configs[3]: synthetic read set, %d reads ~N(10k,1k) samples clipped to [4k,20k] (seed 11), '
                                   'chunksize 4000, overlap 500, batch %d chunks, sharded by read in blocks of %d reads; a step '
                                   '= one pass over the whole read set; random-init weights, head gain %.2f'
                                   % (n_reads, args.batch, B, gain),
                       'reads': n_reads, 'read_samples': total, 'chunks_per_pass': n_chunks,
                       'chunk_samples_per_read_sample': n_chunks * CHUNK / total,
                       'sharding': 'value: blocks k mod G, resident in HBM; e2e: dynamic pull from one shared work queue '
                                   '(process-group store), no data-path collective',
                       'blocks_taken_per_rank_e2e': [r / B / args.steps for r in table['e2e_reads']]},
            'e2e': {'value': total * args.steps / (e2e_ms / 1e3), 'unit': 'samples/s',
                    'h2d_bytes_per_step': int(total * 4), 'd2h_bytes_per_step': int(sum(table['bases']) / args.steps)},
            'gpu_launches': int(sum(table['launches'])),
            'mean_decoded_len_per_read': sum(table['bases']) / args.steps / n_reads,
            # e2e pass, per rank (seconds summed over its blocks; the phases of consecutive blocks overlap): host staging + H2D
            # issue, kernel launches + wait for the letters, string cutting -- against the rank's wall time
            'e2e_phase_seconds_per_rank': {'stage_h2d': table['stage_s'], 'launch_and_wait': table['gpu_s'],
                                           'strings': table['strings_s'], 'wall': [v / 1e3 for v in table['e2e_ms']],
                                           'device_pass': [v / 1e3 for v in table['dev_ms']], 'host_cpus': os.cpu_count()},
            'clocks': clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--dtype', default='fp16', choices=['fp16', 'bf16'])
    ap.add_argument('--batch', type=int, default=BATCH)
    ap.add_argument('--workload', default='chunks', choices=['chunks', 'readset'],
                    help='chunks: BASELINE configs[1] (default, weak scaling); readset: configs[3] (strong scaling)')
    ap.add_argument('--reads', type=int, default=100000)
    ap.add_argument('--block-reads', type=int, default=1024)
    ap.add_argument('--head-gain', type=float, default=None, help='skip the head-gain calibration and use this gain')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-comparator', action='store_true')
    ap.add_argument('--no-train-step', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.workload != 'chunks'):
        ap.error('--dump-outputs is implemented for --impl ours --workload chunks')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if args.workload == 'readset':
        run_readset(args, rank, world, local)
        return

    import torch.distributed as dist
    from oracle import bonito_oracle as bo            # weights generator + cpu_baseline / gpu_comparator legs only
    from xna_basecaller_b200._lib import Handle

    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    N, L, T = args.batch, CHUNK, T_STEPS
    h = Handle(ALPHABET, STATE_LEN, max_N=N, max_T=T, device=dev, bf16=(args.dtype == 'bf16'))
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(N, L, generator=g).pin_memory()
    x_dev = x_host.to(dev)
    sd, head_gain, _ = calibrated_weights(h, bo, x_dev, gain=args.head_gain)
    seq_host = torch.empty(N, T, dtype=torch.int8).pin_memory()
    lens_host = torch.empty(N, dtype=torch.int32).pin_memory()
    seq_dev = torch.empty(N, T, dtype=torch.int8, device=dev)

    def step_device(hh=h):
        return hh.basecall_chunks(x_dev, out=seq_dev)        # fused route: stem, 5 LSTM, head -> exp(scores) -> decode

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed_steps(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), out

    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = h.launches
    dev_ms, (seq, _, lens) = timed_steps(step_device, args.steps)       # the `value` region: no profiling events inside
    launches = h.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'seq': seq, 'lens': lens})     # seq is seq_dev: copied before later steps reuse it
    mean_len = lens.float().mean().item()
    # per-stage device times in a separate, profiled pass of the same steps (CUDA-event spans around every stage)
    h.set_profiling(True)
    h.stage_times()
    timed_steps(step_device, args.steps)
    stages = h.stage_times()
    h.set_profiling(False)

    # end to end through the host-buffer C-ABI call
    # (xb_compute_scores_submit / _wait: the pipelined form of xb_compute_scores_host that basecall() uses -- batch i+1 is
    # submitted before batch i is collected; every step still copies its input from pinned host memory and its result back)
    seq_hosts = [seq_host, torch.empty_like(seq_host).pin_memory()]
    lens_hosts = [lens_host, torch.empty_like(lens_host).pin_memory()]

    def run_e2e(hh, k):
        for i in range(k):
            if i >= 2:
                hh.compute_scores_wait(i & 1)
            hh.compute_scores_submit(i & 1, x_host, seq_hosts[i & 1], lens_hosts[i & 1])
        for i in range(max(k - 2, 0), k):
            hh.compute_scores_wait(i & 1)

    run_e2e(h, 2)
    barrier()
    t0 = time.perf_counter()
    run_e2e(h, args.steps)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    clocks = sampler.summary()

    # the other weight type in the same run (bf16-rounded weights x fp16 activations / fp16 weights), value + e2e
    other = 'bf16' if args.dtype == 'fp16' else 'fp16'
    h2 = Handle(ALPHABET, STATE_LEN, max_N=N, max_T=T, device=dev, bf16=(other == 'bf16'))
    h2.load_weights(sd)
    for _ in range(3):
        step_device(h2)
    other_ms, _ = timed_steps(lambda: step_device(h2), args.steps)
    run_e2e(h2, 2)
    barrier()
    t0 = time.perf_counter()
    run_e2e(h2, args.steps)
    torch.cuda.synchronize(dev)
    other_e2e_s = time.perf_counter() - t0
    h2.close()

    times = torch.tensor([dev_ms, e2e_s * 1e3, other_ms, other_e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, other_ms, other_e2e_ms = times.tolist()
    samples_per_step = N * L * world
    value = samples_per_step * args.steps / (dev_ms / 1e3)
    e2e_value = samples_per_step * args.steps / (e2e_ms / 1e3)

    if rank == 0:
        pk = peaks()
        rec_ms, rec_spans = stages['lstm_recurrence']
        # dominant kernel: the LSTM recurrence (one span = one layer = T recurrent steps of [N,768]x[768,3072])
        flops_per_span = T * 2.0 * N * FEATURES * 4 * FEATURES
        achieved = flops_per_span * rec_spans / (rec_ms / 1e3) / 1e12 if rec_ms > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get('lstm_persistent_kernel', {}).get('dram_bytes_per_launch')

        def stage_ms(*names):
            return sum(stages[k][0] for k in names) / args.steps

        S_BYTES = 4 * h.C * h.NZ
        dec_ms = stage_ms('crf_alpha', 'crf_backward', 'crf_viterbi')
        inproj_ms = stage_ms('lstm_inproj_gemm')
        head_ms = stage_ms('crf_head_gemm')
        conv_ms = stage_ms('conv12_im2col', 'conv3_gemm')
        per_stage = {
            'lstm_inproj_gemm': {'bound': 'tensor', 'achieved': 5 * flops_per_span / (inproj_ms / 1e3) / 1e12,
                                 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s'},
            'crf_head_gemm': {'bound': 'hbm', 'achieved': (T * N * (h.C * h.NZ * 4 + FEATURES * 2)) / (head_ms / 1e3) / 1e9,
                              'peak': pk['hbm_gbs'], 'unit': 'GB/s'},
            'crf_decode': {'bound': 'hbm', 'achieved': (T * N * (2 * S_BYTES + 1)) / (dec_ms / 1e3) / 1e9,
                           'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                           'note': 'algorithmic bytes (2*S+1) per (t, chunk), S = %d B of fp32 scores (SURVEY 8d); the three '
                                   'sweeps actually move 3*S + 7 state vectors of %d B' % (S_BYTES, 4 * (h.C + 7))},
            'conv_stem': {'bound': 'hbm', 'achieved': (N * (L * 4 + T * FEATURES * 2)) / (conv_ms / 1e3) / 1e9,
                          'peak': pk['hbm_gbs'], 'unit': 'GB/s'},
        }
        for v in per_stage.values():
            v['frac'] = v['achieved'] / v['peak']
        line = {
            'metric': 'signal samples/sec basecalled (sup@v3.3 XNA)', 'value': value, 'unit': 'samples/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': dev_ms / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
            'config': dict(workload_config(N, L), head_gain=head_gain),
            'e2e': {'value': e2e_value, 'unit': 'samples/s', 'h2d_bytes_per_step': N * L * 4 * world,
                    'd2h_bytes_per_step': (N * T + N * 4) * world},
            'gpu_launches': launches,
            'mean_decoded_len': mean_len,
            'roofline': {'bound': 'tensor', 'kernel': 'lstm_recurrence', 'achieved': achieved, 'peak': pk['tf_sustained'],
                         'unit': 'TFLOP/s', 'frac': achieved / pk['tf_sustained'], 'traffic': traffic,
                         'peak_source': pk['source'] + ', sustained figure (kernel timed inside a long step)'},
            'stage_rooflines': per_stage,
            'stages_ms_per_step': {k: v[0] / args.steps for k, v in stages.items()},
            'model_tflops': (sum(FLOP_PER_CHUNK.values()) * N * world) / (dev_ms / args.steps / 1e3) / 1e12,
            'clocks': clocks,
            'other_dtype': {'dtype': other, 'value': samples_per_step * args.steps / (other_ms / 1e3),
                            'ms_per_step': other_ms / args.steps,
                            'e2e': samples_per_step * args.steps / (other_e2e_ms / 1e3), 'unit': 'samples/s'},
        }
        if world == 1 and not args.no_gpu_comparator:
            try:
                line['gpu_comparator'] = gpu_comparator(sd, dev, N)
            except Exception as e:                                    # a baseline leg must not take the bench line down
                line['gpu_comparator'] = {'unavailable': repr(e)[:200]}
        if world == 1 and not args.no_train_step:
            try:
                line['train_step'] = train_step_leg(dev, N)
            except Exception as e:                                    # a side leg must not take the bench line down
                line['train_step'] = {'unavailable': repr(e)[:200]}
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            n_chunks = 64                             # = BASELINE.json configs[0]
            cpu_reference_pass(4, cores)
            sec = cpu_reference_pass(n_chunks, cores, repeats=2)
            line['cpu_baseline'] = {'value': n_chunks * L / sec, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                                    'sample': '%d chunks x %d samples, best of 2 (torch fp32 encoder + C CRF decode, both on '
                                              'all %d host threads)' % (n_chunks, L, cores)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
