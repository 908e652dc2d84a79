#!/usr/bin/env python
"""bench.py — questions/sec of the N2NMN module-network hot path on B200 (BASELINE.json metric).

One step = one pass of the hot path over one batch of synthetic input (default workload: CLEVR
gt-layout eval, 64 questions, 10x15x512 pool5 grid, T=20 layout tokens, expert-layout mix): host
layout compile (C++) -> table upload -> text projection -> tcgen05 conv_image contraction with the
fused Find epilogue -> tree kernel -> scores [64,28] on device. Inputs come from a pool of distinct
batches resident in HBM that is larger than L2, walked round-robin, so no step re-reads a cached
batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config clevr|shapes|vqa514|vqa2050|stress]
    python bench.py --impl reference ...        # CPU arm (the oracle restatement of the reference)

How the number is taken: --warmup W steps, then exactly --steps K timed steps, queued back to back
on the executor pool and walking the resident batches round-robin. The warm-up is queued right
before the timed steps, so the pool's worker threads and streams are already running when the
timed steps begin; CUDA events on the current stream bracket the K timed steps only. A step takes
~10 us on a B200 (1000 W power limit), so K in the thousands keeps the fill and drain of the pool's
streams and host noise out of the number (measured there with W=20: 5.6-5.8 M questions/s at
K=200, 6.4 M at K=4000). Under torchrun every rank owns one GPU and its own shard of the questions
(weak scaling, no data-path collective: questions are independent, SURVEY.md §8e); region time =
max over ranks; rank 0 prints ONE JSON line.

`--dump-outputs DIR` writes what the last timed step computed (rank 0's shard) as DIR/scores.npy
(float32 [B, C]) and DIR/validity.npy (float32 [B], 1 = the layout assembled). Inputs, weights and
layouts are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TEXT_DIM = 300
UNIT = 'questions/s'
# mma.sync.m16n8k8.tf32 issues once per ~36 cycles per SM sub-partition on this part (measured:
# tools/ubench/mma_tf32.cu, DESIGN.md §4): 4 x 2048 flop / 36 clk x 148 SMs x 1.965 GHz. The
# ceiling of every mma.sync kernel here (the fp32-parity text / quad products run 3 passes).
MMA_SYNC_TF32_TFLOPS = 4 * 2048 / 36.0 * 148 * 1.965e9 / 1e12

# BASELINE.json configs made concrete (SURVEY.md §0 table, §8d). `clevr` is the configuration the
# metric is quoted on; the others are reported beside it (`other_configs`) or with --config.
WORKLOADS = {
    'clevr': dict(family='clevr', B=64, H=10, W=15, D=512, T=20, C=28, layouts='expert',
                  metric='clevr_questions_per_sec',
                  title='CLEVR gt-layout eval, batch=64/GPU, 10x15x512 pool5, %s layouts depth<=12, T=20'),
    'shapes': dict(family='shapes', B=32, H=3, W=3, D=64, T=11, C=2, layouts='shapes_hist',
                   metric='shapes_questions_per_sec',
                   title='SHAPES gt-layout eval, batch=32/GPU, 3x3x64 conv features, %s layouts, T=11'),
    'vqa514': dict(family='vqa', B=128, H=14, W=14, D=512, T=13, C=3001, layouts='vqa_hist',
                   metric='vqa_questions_per_sec',
                   title='VQA gt-layout eval, batch=128/GPU, 14x14x512(+2 coord) features, %s layouts, T=13'),
    'vqa2050': dict(family='vqa', B=128, H=14, W=14, D=2048, T=13, C=3001, layouts='vqa_hist',
                    metric='vqa_questions_per_sec',
                    title='VQA gt-layout eval, batch=128/GPU, 14x14x2048(+2 coord) res5c features, %s layouts, T=13'),
    'stress': dict(family='clevr', B=128, H=20, W=20, D=1024, T=40, C=28, layouts='deep16',
                   metric='stress_questions_per_sec',
                   title='synthetic stress, batch=128/GPU, 20x20x1024 features, %s layouts depth<=16, T=40'),
}
L2_BYTES = 126e6


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200, help='timed steps')
    ap.add_argument('--warmup', type=int, default=20, help='untimed steps before them')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write the last timed step\'s scores / validity to DIR/<name>.npy')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='clevr', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0, help='questions per GPU per step (0 = the config\'s)')
    ap.add_argument('--layouts', default=None, choices=['expert', 'random', 'deep'],
                    help='CLEVR layout set (default expert)')
    ap.add_argument('--min-seconds', type=float, default=0.5, help='ignored (old command lines)')
    ap.add_argument('--trials', type=int, default=3, help='ignored (old command lines)')
    ap.add_argument('--cpu-seconds', type=float, default=10.0, help='cpu_baseline sample budget')
    ap.add_argument('--ref-seconds', type=float, default=0.0,
                    help='--impl reference: stop after this many seconds (0 = run all --steps)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--wave', action='store_true', help='depth-bucketed wave executor')
    ap.add_argument('--no-train', action='store_true', help='skip the train-step measurement')
    ap.add_argument('--no-seq2seq', action='store_true',
                    help='skip the layout-generator (seq2seq, SURVEY §8 f1) measurement')
    ap.add_argument('--no-other-sets', action='store_true',
                    help='skip the random / deep layout sets reported beside the expert mix')
    ap.add_argument('--no-other-configs', action='store_true',
                    help='skip the other BASELINE.json workloads reported beside the headline')
    ap.add_argument('--tree-cluster', type=int, default=None,
                    help='CTAs per question in the executor kernel (default: chosen by the pool)')
    ap.add_argument('--proj-ctas', type=int, default=None,
                    help='cap of the contraction kernel grid (default: chosen by the pool; 0 = all SMs)')
    ap.add_argument('--streams', type=int, default=0,
                    help='contexts/streams/worker threads (0 = the library default)')
    ap.add_argument('--host-threads', type=int, default=0, help='ignored (old command lines)')
    ap.add_argument('--pool', type=int, default=0, help='ignored (old command lines)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    return args


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'],
                    bf16_sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0,
                source='fallback (B200_PROFILING.md)')


def ncu_traffic(kernel, batches_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed
    `ncu --set full` capture of this same command (profiles/ncu_traffic.json); None when there
    is no capture or it was taken with another number of batches per launch."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if not os.path.exists(p):
        return None
    with open(p) as f:
        d = json.load(f).get(kernel)
    if not d or d.get('batches_per_launch', 8) != batches_per_launch:
        return None
    return d['dram_read_bytes'] + d['dram_write_bytes']


def workload_title(wl, layouts):
    names = {'expert': 'expert', 'random': 'random valid', 'deep': 'deep', 'shapes_hist':
             'the 3 real SHAPES', 'vqa_hist': 'VQA gt-layout histogram', 'deep16': 'random deep'}
    return wl['title'] % names[layouts]


def make_tokens(asm, kind, n, T, seed):
    from n2nmn_b200 import synth
    rng = np.random.RandomState(seed)
    if kind == 'expert':
        toks = synth.expert_mix_tokens(asm, n, T)       # same mix, different question order
        return np.ascontiguousarray(toks[:, rng.permutation(n)])
    if kind == 'random':
        return synth.random_valid_tokens(asm, n, T, seed=seed)
    if kind == 'deep':
        return synth.random_valid_tokens(asm, n, T, seed=seed, ans_weight=0.15, min_depth=3,
                                         max_depth=12)
    if kind == 'shapes_hist':
        return synth.histogram_tokens(asm, synth.SHAPES_LAYOUTS, n, T, seed=seed)
    if kind == 'vqa_hist':
        return synth.histogram_tokens(asm, synth.VQA_LAYOUTS, n, T, seed=seed)
    if kind == 'deep16':   # sampling by rejection is slow: 16 distinct deep layouts, tiled
        base = synth.random_valid_tokens(asm, 16, T, seed=21, ans_weight=0.08, min_depth=8,
                                         max_depth=16)
        return np.ascontiguousarray(base[:, rng.randint(0, 16, size=n)])
    raise ValueError(kind)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md): one
    `nvidia-smi -lms` process started right before the region and stopped right after it."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '20'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)      # let the first samples start flowing
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                out = ''
            rows = [[c.strip() for c in ln.split(',')] for ln in out.splitlines() if ln.strip()]
        sm = [float(r[1]) for r in rows if len(r) > 2 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace('.', '').isdigit()]
        pw = [float(r[3]) for r in rows if len(r) > 3 and r[3].replace('.', '').isdigit()]
        reasons = []
        for name, col in (('hw_slowdown', 4), ('hw_thermal_slowdown', 5),
                          ('sw_thermal_slowdown', 6), ('sw_power_cap', 7)):
            if any(len(r) > col and r[col].lower().startswith('active') for r in rows):
                reasons.append(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'power_w_max': max(pw) if pw else None, 'samples': len(rows)}


# =========================================================================== CPU arms (oracle)
def _thread_candidates():
    # (one thread per hardware thread was measured pathological on the 128-cpu box: 5.8 s per
    # batch with torch, 0.2-0.3 s with OpenBLAS, against 8-40 ms at 16-32 threads)
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    return sorted({min(ncpu, c) for c in (8, 16, 32, 64)})


class CpuPort:
    """One CPU restatement of the reference path (TF 1.0 + Fold cannot be installed here,
    DESIGN.md): Assembler.assemble + depth-batched module calls. kind 'numpy' = oracle/nmn_oracle.py
    (numpy + OpenBLAS), kind 'torch' = oracle/nmn_oracle_torch.py::run_depth_batched (MKL/oneDNN)."""

    def __init__(self, kind, wl, feat, word_vecs, weights):
        from n2nmn_b200 import synth
        from n2nmn_b200.assembler import Assembler
        self.kind = kind
        self.asm = Assembler(synth.vocab_file(wl['family']))
        if kind == 'numpy':
            from oracle.nmn_oracle import OracleModules, run_depth_batched
            self.m = OracleModules(feat, word_vecs, wl['C'], weights, family=wl['family'])
            self.run = run_depth_batched
        else:
            from oracle import nmn_oracle_torch as ot
            self.m = ot.TorchOracleModules(feat, word_vecs, wl['C'], weights, family=wl['family'])
            self.run = ot.run_depth_batched
        self.threads = None

    def step(self, tokens):
        exprs, _ = self.asm.assemble(tokens)
        return self.run(self.m, exprs)

    def set_threads(self, nt):
        if self.kind == 'torch':
            import torch
            torch.set_num_threads(int(nt))
        else:
            from threadpoolctl import threadpool_limits
            if getattr(self, '_lim', None) is not None:
                self._lim.restore_original_limits()
            self._lim = threadpool_limits(limits=int(nt))
        self.threads = int(nt)

    def pick_threads(self, tokens, trials=3, max_seconds=6.0):
        """One thread per core is slow on many-core hosts for these small GEMMs, and one noisy
        trial picked a 2x slower count in round 1: median of `trials` per candidate."""
        best, t_start = (None, None), time.perf_counter()
        log = {}
        for nt in _thread_candidates():
            self.set_threads(nt)
            self.step(tokens)
            self.step(tokens)
            ts = []
            for _ in range(trials):
                t0 = time.perf_counter()
                self.step(tokens)
                ts.append(time.perf_counter() - t0)
            med = float(np.median(ts))
            log[nt] = round(med * 1e3, 2)
            if best[0] is None or med < best[0]:
                best = (med, nt)
            if time.perf_counter() - t_start > max_seconds and best[0] is not None:
                break
        self.set_threads(best[1])
        self.pick_log = log
        return best[1]

    def measure(self, tokens_list, budget_s, min_batches=2):
        n_q, t0, k = 0, time.perf_counter(), 0
        while True:
            tok = tokens_list[k % len(tokens_list)]
            self.step(tok)
            n_q += tok.shape[1]
            k += 1
            el = time.perf_counter() - t0
            if k >= min_batches and el >= budget_s:
                break
        return n_q / el, k, el


def best_cpu_port(wl, feat, word_vecs, weights, toks, pick_seconds=6.0):
    """Both ports with their best thread count; returns (faster port, {kind: ms per batch})."""
    ports, ms = [], {}
    for kind in ('numpy', 'torch'):
        try:
            p = CpuPort(kind, wl, feat, word_vecs, weights)
            p.pick_threads(toks[0], max_seconds=pick_seconds)
            for i in range(3):   # settle on the chosen thread count before timing
                p.step(toks[i % len(toks)])
            t0 = time.perf_counter()
            for i in range(4):
                p.step(toks[i % len(toks)])
            ms[kind] = {'ms_per_batch': round((time.perf_counter() - t0) * 250, 2),
                        'threads': p.threads, 'ms_by_threads': p.pick_log}
            ports.append(p)
        except Exception as e:   # threadpoolctl / torch missing: keep the other port
            ms[kind] = {'error': repr(e)}
    best = min(ports, key=lambda p: ms[p.kind]['ms_per_batch'])
    best.set_threads(best.threads)
    return best, ms


def port_desc(p):
    return ('oracle/nmn_oracle.py: numpy+OpenBLAS' if p.kind == 'numpy' else
            'oracle/nmn_oracle_torch.py: torch-CPU MKL/oneDNN') + \
        ' fp32 depth-batched restatement, Assembler.assemble included'


def run_reference_arm(args, rank, world):
    """--impl reference: the faster CPU restatement (oracle) of the reference's TF1 path on the
    box's host cores, same workload/config strings as the b200 arm. Rank 0 only."""
    if rank != 0:
        return
    try:   # all host cores, whatever the launcher (or a parent GPU arm bound to a NUMA node) set
        os.sched_setaffinity(0, range(os.cpu_count()))
    except Exception:
        pass
    from n2nmn_b200 import synth, weights as wts
    from n2nmn_b200.assembler import Assembler
    wl = dict(WORKLOADS[args.config])
    B = args.batch or wl['B']
    layouts = args.layouts or wl['layouts']
    asm = Assembler(synth.vocab_file(wl['family']))
    feat, word_vecs = synth.make_inputs(B, wl['H'], wl['W'], wl['D'], wl['T'], seed=1234)
    weights = wts.init_weights(wl['family'], wl['H'], wl['W'], wl['D'], wl['C'], seed=0,
                               bias_std=0.1)
    toks = [make_tokens(asm, layouts, B, wl['T'], seed=100 + i) for i in range(4)]
    port, ports_ms = best_cpu_port(wl, feat, word_vecs, weights, toks)
    for i in range(max(args.warmup, 1)):
        port.step(toks[i % 4])
    steps = args.steps
    per = []
    t0 = time.perf_counter()
    for i in range(steps):
        t1 = time.perf_counter()
        port.step(toks[i % 4])
        per.append(time.perf_counter() - t1)
        if args.ref_seconds > 0 and time.perf_counter() - t0 > args.ref_seconds and i >= 1:
            steps = i + 1      # bounded sample (big workloads: seconds per batch)
            break
    el = time.perf_counter() - t0
    # The CPU arm's step time is bimodal on the many-core box (median 7.6 ms, mean 14-17 ms: a few
    # steps of > 100 ms, allocator / thread-pool hiccups of the CPU libraries), which made the
    # baseline differ by 20 % between two runs of the same command. The MEDIAN step is what is
    # reported: it is the stable figure and the one that favours the reference.
    med = float(np.median(per))
    qps = B / med
    line = {
        'impl': 'reference', 'metric': wl['metric'], 'value': qps, 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * med, 'mean_ms_per_step': 1e3 * el / steps,
        'median_ms_per_step': 1e3 * med, 'value_from_mean': steps * B / el,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': workload_title(wl, layouts), 'global_batch': B},
        'cpu_baseline': {'value': qps, 'unit': UNIT, 'cores': port.threads, 'kind': 'port',
                         'host_cpus': os.cpu_count(), 'ports': ports_ms,
                         'sample': '%d batches of %d questions (%s)' % (steps, B, port_desc(port))},
        'e2e': {'value': qps, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    if args.config == 'clevr' and not args.no_seq2seq:
        line['cpu_baseline']['layout_generator'] = seq2seq_cpu_port(asm, B)
    print(json.dumps(line), flush=True)


SEQ2SEQ = dict(T_encoder=45, T_decoder=20, num_vocab_txt=90, embed_dim=300, lstm_dim=512,
               num_layers=2)   # exp_clevr/train_clevr_gt_layout.py:22-40


def seq2seq_inputs(B, seed=0):
    rng = np.random.RandomState(seed)
    seq = rng.randint(0, SEQ2SEQ['num_vocab_txt'], size=(SEQ2SEQ['T_encoder'], B)).astype(np.int32)
    lens = rng.randint(5, SEQ2SEQ['T_encoder'] + 1, size=B).astype(np.int32)
    return seq, lens


def seq2seq_measure(torch, asm, dev, B, reps=30):
    from n2nmn_b200.seq2seq import AttentionSeq2Seq
    from n2nmn_b200.weights import init_seq2seq_weights
    c = SEQ2SEQ
    w = init_seq2seq_weights(c['num_vocab_txt'], c['embed_dim'], asm.num_vocab_nmn, c['embed_dim'],
                             c['lstm_dim'], c['num_layers'])
    s = AttentionSeq2Seq(None, None, c['T_decoder'], c['num_vocab_txt'], c['embed_dim'],
                         asm.num_vocab_nmn, c['embed_dim'], c['lstm_dim'], c['num_layers'], asm,
                         T_encoder=c['T_encoder'], max_batch=B, weights=w, device=dev)
    seq, lens = seq2seq_inputs(B)
    seq, lens = torch.from_numpy(seq).to(dev), torch.from_numpy(lens).to(dev)
    for _ in range(5):
        s.forward(seq, lens)
    torch.cuda.synchronize()
    n0 = s.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        s.forward(seq, lens)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return {'what': 'AttentionSeq2Seq forward (encoder LSTM x%d, attention decoder, greedy), '
                    'N=%d T_encoder=%d T_decoder=%d lstm_dim=%d; fp32 via 3xTF32 mma.sync'
                    % (c['num_layers'], B, c['T_encoder'], c['T_decoder'], c['lstm_dim']),
            'ms_per_batch': ms, 'questions_per_sec': B / (ms * 1e-3),
            'gpu_launches_per_batch': (s.launch_count() - n0) // reps, 'reps': reps}


def seq2seq_cpu_port(asm, B):
    """The numpy restatement of the layout generator, timed once (cpu_baseline leg only)."""
    from oracle import seq2seq_oracle as so
    from n2nmn_b200.weights import init_seq2seq_weights
    c = SEQ2SEQ
    w = init_seq2seq_weights(c['num_vocab_txt'], c['embed_dim'], asm.num_vocab_nmn, c['embed_dim'],
                             c['lstm_dim'], c['num_layers'])
    seq, lens = seq2seq_inputs(B)
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        so.run(w, seq, lens, c['T_decoder'], c['num_layers'], asm.P, asm.W, asm.b)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {'ms_per_batch': 1e3 * best, 'questions_per_sec': B / best, 'kind': 'port (numpy/BLAS)',
            'sample': '1 batch of %d questions, best of 2' % B}


# =========================================================================== GPU arm
def bind_to_gpu_numa_node(torch, index):
    """Run this process (and so its pinned-buffer allocations and the pool's worker threads) on
    the CPUs that are local to the GPU's PCIe root: host<->device copies from the other socket
    run at about half the rate on a two-socket box. Best effort; returns what was done."""
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = '%04x:%02x:%02x.0' % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open('/sys/bus/pci/devices/%s/local_cpulist' % bdf) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(','):
            if '-' in part:
                a, b = part.split('-')
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return 'no local cpus in the affinity mask'
        os.sched_setaffinity(0, cpus)
        return 'bound to %d cpus local to %s (%s)' % (len(cpus), bdf, spec)
    except Exception as e:   # no sysfs in this container, or not a PCI device
        return 'not bound: %s' % e


class Bench:
    """One workload on this rank's GPU: resident batches, the executor pool, timed regions."""

    def __init__(self, torch, dist, args, wl, layouts, B, rank, world, dev, streams=None,
                 device_synth=False):
        from n2nmn_b200 import _lib, synth, weights as wts
        from n2nmn_b200.assembler import Assembler
        from n2nmn_b200.executor import ExecutorPool
        self.torch, self.dist, self.args, self.wl = torch, dist, args, wl
        self.rank, self.world, self.dev, self.B, self.layouts = rank, world, dev, B, layouts
        H, W, D, T, C = wl['H'], wl['W'], wl['D'], wl['T'], wl['C']
        self.asm = Assembler(synth.vocab_file(wl['family']))
        self.weights = wts.init_weights(wl['family'], H, W, D, C, seed=0, bias_std=0.1)
        batch_bytes = B * H * W * D * 4
        self.P = P = int(min(2048, max(2, math.ceil(1.5 * L2_BYTES / batch_bytes))))
        self.batch_bytes = batch_bytes
        self.feats, self.wvs = [], []
        for i in range(P):   # per-rank seeds = per-rank shard of the global question stream
            seed = 1234 + 1000 * rank + i
            if device_synth:   # big grids: generate on the device (same distributions)
                g = torch.Generator(device=dev)
                g.manual_seed(seed)
                f = torch.randn((B, H, W, D), generator=g, device=dev).clamp_(min=0)
                w = torch.randn((T, B, TEXT_DIM), generator=g, device=dev).mul_(0.3)
            else:
                fn, wn = synth.make_inputs(B, H, W, D, T, seed=seed)
                f, w = torch.from_numpy(fn).to(dev), torch.from_numpy(wn).to(dev)
            self.feats.append(f)
            self.wvs.append(w)
        n_tok = min(P, 16)
        self.toks = [make_tokens(self.asm, layouts, B, T, seed=100 + 1000 * rank + i)
                     for i in range(n_tok)]
        kw = {}
        if streams:
            kw['num_streams'] = streams
        flags = _lib.FLAG_WAVE_EXECUTOR if args.wave else 0
        self.pool = ExecutorPool(wl['family'], self.feats[0], self.wvs[0], C, self.asm,
                                 weights=self.weights, flags=flags, max_batch=B, max_T=T,
                                 tree_cluster=args.tree_cluster, proj_ctas=args.proj_ctas, **kw)
        self.K = len(self.pool)
        self.ex = self.pool.executors[0]
        self.nout = max(2 * self.K, 8)
        self.outs = [torch.empty((B, C), dtype=torch.float32, device=dev) for _ in range(self.nout)]

    def tok(self, i):
        return self.toks[i % len(self.toks)]

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def allmax(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def block(self, first, n, toks=None, outs=None):
        """Pre-marshalled steps first .. first+n-1 of the round-robin walk over the resident
        batches; score buffers from the ring `self.outs` unless `outs` is given."""
        toks = toks or self.toks
        idx = [(first + j) % self.P for j in range(n)]
        outs = outs or [self.outs[(first + j) % self.nout] for j in range(n)]
        return self.pool.make_block([self.feats[i] for i in idx], [self.wvs[i] for i in idx],
                                    [toks[i % len(toks)] for i in idx], outs)

    def blocks(self, steps, toks=None):
        """Pre-marshalled blocks of `steps` steps that together walk all P resident batches."""
        nb = min(64, self.P // math.gcd(steps, self.P))
        return [self.block(b * steps, steps, toks) for b in range(nb)]

    def headline(self, steps, warmup):
        """`warmup` steps, then exactly `steps` timed steps. The warm-up is queued right before
        the timed steps, so the timed steps start with the pool's worker threads running; CUDA
        events bracket the timed steps only. Returns the timing and what the last timed step
        computed: scores [B, C] float32 and validity bool[B]. That step writes a buffer of its
        own: the ring `self.outs` is shared by steps of one launch group."""
        torch = self.torch
        last = torch.empty((self.B, self.wl['C']), dtype=torch.float32, device=self.dev)
        outs = [self.outs[(warmup + j) % self.nout] for j in range(steps - 1)] + [last]
        blk = self.block(warmup, steps, outs=outs)
        warm = self.block(0, warmup) if warmup > 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        if warm is not None:
            self.pool.begin()
            self.pool.submit_block(warm)
            self.pool.end()
        l0 = self.pool.launch_count()
        e0.record()
        t0 = time.perf_counter()
        self.pool.begin()
        valid = self.pool.submit_block(blk)
        self.pool.end()
        e1.record()
        host_ms = (time.perf_counter() - t0) * 1e3
        self.barrier()
        ms = self.allmax(e0.elapsed_time(e1))
        return {'ms_per_step': ms / steps, 'timed_steps': steps,
                'gpu_launches': self.pool.launch_count() - l0, 'timed_region_s': ms * 1e-3,
                'host_enqueue_ms_per_step': host_ms / steps,
                'value': self.world * self.B * steps / (ms * 1e-3),
                'scores': last.cpu().numpy(), 'validity': valid[steps - 1].astype(bool)}

    def region(self, blocks, repeats):
        """`repeats` back-to-back repetitions of the step block, CUDA events on the current stream
        (pool.begin()/end() order the pool's streams after e0 / before e1). Returns ms, max over
        ranks, and the host time needed to enqueue."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        t0 = time.perf_counter()
        self.pool.begin()
        for r in range(repeats):
            self.pool.submit_block(blocks[r % len(blocks)])
        self.pool.end()
        e1.record()
        host_ms = (time.perf_counter() - t0) * 1e3
        self.barrier()
        return self.allmax(e0.elapsed_time(e1)), host_ms

    def timed(self, steps, warmup, min_seconds, trials, toks=None):
        """warm-up, calibration, then `trials` regions of >= min_seconds; median region reported."""
        if warmup > 0:
            wb = self.blocks(warmup, toks)
            self.region(wb[:1], 1)
        blocks = self.blocks(steps, toks)
        cal_ms, _ = self.region(blocks, max(1, len(blocks)))      # touches every resident batch
        per_block = cal_ms / max(1, len(blocks))
        # the first estimate includes the pipeline fill of a short region: refine it on ~15 % of
        # the target length before fixing the number of repetitions
        R1 = int(max(1, math.ceil(0.15 * min_seconds * 1e3 / max(per_block, 1e-6))))
        cal_ms, _ = self.region(blocks, R1)
        per_block = cal_ms / R1
        R = int(max(1, math.ceil(min_seconds * 1e3 / max(per_block, 1e-6))))
        res = []
        for _ in range(trials):
            l0 = self.pool.launch_count()
            ms, host_ms = self.region(blocks, R)
            res.append((ms, host_ms, self.pool.launch_count() - l0))
        res.sort()
        ms, host_ms, launches = res[len(res) // 2]
        n_steps = R * steps
        return {'ms_per_step': ms / n_steps, 'repeats': R, 'timed_steps': n_steps,
                'gpu_launches': int(launches),
                'timed_region_s': ms * 1e-3, 'host_enqueue_ms_per_step': host_ms / n_steps,
                'value': self.world * self.B * n_steps / (ms * 1e-3),
                'trial_values': [self.world * self.B * n_steps / (r[0] * 1e-3) for r in res]}

    def kernel_pass(self, n=30):
        """Per-launch CUDA events (library profiling mode) of the kernels AS LAUNCHED IN THE TIMED
        REGION: one context evaluating groups of `max_group` batches per set of launches
        (n2nmn_forward_group), walking the resident batches: {kernel: mean us per launch}, mean
        algorithmic bytes / flops per launch of each of the three kernels (SURVEY.md §8d)."""
        ex, acc, nb, nf = self.ex, {}, np.zeros(3), np.zeros(3)
        G = self.pool.max_group
        name2idx = self.asm.name2idx_dict
        pooled_w = {name2idx[k]: v for k, v in (('_Describe', 1), ('_SameProperty', 2))
                    if k in name2idx}
        self.pooled_roots = 0.0     # mean pooled answer roots per launch (pool_kernel's work)
        outs = [self.outs[g % self.nout] for g in range(G)] if G > self.nout else self.outs[:G]

        def run(i):
            idx = [(i * G + g) % self.P for g in range(G)]
            ex.forward_group([self.feats[j] for j in idx], [self.wvs[j] for j in idx],
                             [self.tok(j) for j in idx], outs=outs)
        for i in range(3):
            run(i)
        ex.set_profiling(True)
        for i in range(n):
            run(i)
            for name, us in ex.launch_times():
                acc.setdefault(name, []).append(us)
            info = ex.last_step_info()
            for g in range(G):
                tk = self.tok((i * G + g) % self.P)
                self.pooled_roots += sum(w * int((tk == t).sum()) for t, w in pooled_w.items()) / n
            nb += np.array(info['kernel_bytes'], float)
            nf += np.array(info['kernel_flops'], float)
        ex.set_profiling(False)
        return {k: float(np.mean(v)) for k, v in acc.items()}, nb / n, nf / n

    def roofline(self, pk):
        """roofline of the dominant kernel (the contraction) + HBM fractions of the other two."""
        kus, nb, nf = self.kernel_pass()
        tf32_peak = pk['bf16_tflops'] / 2
        total = max(sum(kus.values()), 1e-9)

        def frac(us, b, f):
            d = us * 1e-6
            return b / d / 1e9, f / d / 1e12, b / d / 1e9 / pk['hbm_gbs'], f / d / 1e12 / tf32_peak

        out = {'kernel_us': kus}
        proj = 'proj_umma_kernel'
        if proj in kus:
            gbs, tfs, hf, tf = frac(kus[proj], nb[1], nf[1])
            bound = 'hbm' if hf >= tf else 'tensor'
            out['roofline'] = {
                'kernel': proj, 'bound': bound, 'achieved': gbs if bound == 'hbm' else tfs,
                'peak': pk['hbm_gbs'] if bound == 'hbm' else tf32_peak,
                'unit': 'GB/s' if bound == 'hbm' else 'TFLOP/s', 'frac': max(hf, tf),
                'traffic': (ncu_traffic(proj, self.pool.max_group) if self.wl is WORKLOADS['clevr']
                            else None),
                'hbm_frac': hf, 'tensor_frac_of_tf32_peak': tf, 'avg_launch_us': kus[proj],
                'algorithmic_bytes_per_launch': nb[1], 'flops_per_launch': nf[1],
                'peak_source': pk['source'] + '; TF32 peak taken as bf16 burst / 2',
                'share_of_step': kus[proj] / total,
                'batches_per_launch': self.pool.max_group,
                'how': 'CUDA events around every launch (library profiling mode), one context '
                       'running groups of %d batches per launch as the pool does in the timed '
                       'region, mean of 30 groups over the resident batches'
                       % self.pool.max_group}
        for key, name, k in (('roofline_text', 'text_proj_kernel', 0),
                             ('roofline_tree', 'tree_kernel', 2)):
            if name in kus:
                gbs, tfs, hf, tf = frac(kus[name], nb[k], nf[k])
                out[key] = {'kernel': name, 'bound': 'hbm', 'achieved': gbs, 'peak': pk['hbm_gbs'],
                            'unit': 'GB/s', 'frac': hf, 'avg_launch_us': kus[name],
                            'algorithmic_bytes_per_launch': nb[k], 'flops_per_launch': nf[k],
                            'batches_per_launch': self.pool.max_group,
                            'share_of_step': kus[name] / total}
        try:    # derived figures; never allowed to cost the line
            if self.wl is WORKLOADS['clevr'] and 'roofline_text' in out:
                # the text kernel's governing limit is the mma.sync issue rate, not HBM: three
                # error-compensated TF32 passes over [rows, 304] x [304, 256] (K, M padded)
                r = out['roofline_text']
                rows = nf[0] / (2.0 * TEXT_DIM * 250)
                issued = 3 * 2.0 * rows * 304 * 256
                tf = issued / (r['avg_launch_us'] * 1e-6) / 1e12
                r['issue_rate'] = {'bound': 'mma.sync issue rate (fp32-parity 3xTF32)',
                                   'issued_flops_per_launch': issued, 'achieved': tf,
                                   'peak': MMA_SYNC_TF32_TFLOPS, 'unit': 'TFLOP/s',
                                   'frac': tf / MMA_SYNC_TF32_TFLOPS, 'rows_per_launch': rows}
            if self.wl['family'] == 'clevr' and 'pool_kernel' in kus and self.pooled_roots > 0:
                b = self.pooled_roots * self.wl['H'] * self.wl['W'] * self.wl['D'] * 4.0
                gbs = b / (kus['pool_kernel'] * 1e-6) / 1e9
                out['roofline_pool'] = {
                    'kernel': 'pool_kernel', 'bound': 'hbm', 'achieved': gbs,
                    'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / pk['hbm_gbs'],
                    'avg_launch_us': kus['pool_kernel'], 'algorithmic_bytes_per_launch': b,
                    'pooled_roots_per_launch': self.pooled_roots,
                    'traffic': ncu_traffic('pool_kernel', self.pool.max_group),
                    'batches_per_launch': self.pool.max_group,
                    'share_of_step': kus['pool_kernel'] / total,
                    'note': 'algorithmic = one H*W*D feature grid per pooled root (Describe 1, '
                            'SameProperty 2); grids the contraction has just read are partly '
                            'served from L2 (traffic = DRAM bytes of the ncu capture)'}
        except Exception as e:   # noqa: BLE001
            out['roofline_derived_error'] = repr(e)
        return out

    def e2e(self, steps, min_seconds, feat_f16=False):
        """Pinned host features + word vectors -> H2D -> kernels -> D2H scores, every step, through
        ExecutorPool (n2nmn_forward_host_async per step); wall clock + final synchronize.
        feat_f16: the feature grids are stored as fp16 on the host (a secondary number: not the
        reference's fp32 feed; n2nmn_forward_group_host_f16_async widens them on the device)."""
        torch = self.torch
        hp = int(min(self.P, max(2, math.ceil(1.2 * L2_BYTES / self.batch_bytes)), 8))
        hf = [(self.feats[i].half() if feat_f16 else self.feats[i]).cpu().pin_memory()
              for i in range(hp)]
        hw = [self.wvs[i].cpu().pin_memory() for i in range(hp)]
        # one score buffer per host batch: steps that share a buffer have identical inputs
        hs = [torch.empty((self.B, self.wl['C']), dtype=torch.float32).pin_memory()
              for _ in range(hp)]
        k = max(hp, min(steps, 50))
        idx = [j % hp for j in range(k)]
        blk = self.pool.make_block([hf[i] for i in idx], [hw[i] for i in idx],
                                   [self.tok(i) for i in idx], [hs[i] for i in idx],
                                   host_io=True)

        def run(reps):
            self.barrier()
            t0 = time.perf_counter()
            self.pool.begin()
            for _ in range(reps):
                self.pool.submit_block(blk)
            self.pool.end()
            torch.cuda.synchronize()
            return self.allmax(time.perf_counter() - t0)

        run(1)
        cal = run(1)
        reps = int(max(1, math.ceil(min_seconds / max(cal, 1e-6))))
        els = sorted(run(reps) for _ in range(3))
        el = els[1]
        # the copied-back scores are the device path's scores
        last = k - 1
        chk, _ = self.ex.forward_device(self.feats[idx[last]], self.wvs[idx[last]],
                                        self.tok(idx[last]))
        torch.cuda.synchronize()
        diff = float((hs[idx[last]] - chk.cpu()).abs().max())
        if feat_f16:
            assert diff <= 1e-3, 'fp16-feature e2e scores differ from the fp32 feed by %g' % diff
        else:
            assert diff == 0.0, 'e2e scores differ from the device path'
        h2d = int(hf[0].numel() * hf[0].element_size() + hw[0].numel() * 4)
        d2h = int(hs[0].numel() * 4)
        n = reps * k
        return {'value': self.world * self.B * n / el, 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'steps': n, 'timed_region_s': el,
                'bound': 'pcie', 'achieved_h2d_gbs_per_gpu': h2d * n / el / 1e9,
                'host_feature_dtype': 'f16' if feat_f16 else 'f32',
                'max_abs_score_diff_vs_f32_device_path': diff,
                'how': 'ExecutorPool.submit_block(host_io): pinned host features+word_vecs -> '
                       'async H2D -> C++ layout compile -> kernels -> async D2H scores, %d '
                       'streams, every step; wall clock around the loop + final synchronize, '
                       'median of 3 regions' % self.K}

    def cpu_baseline(self, budget_s, config):
        """The reference arm (`bench.py --impl reference`) in a subprocess on a bounded sample:
        the same code path and process conditions (all host cores, no CUDA context, no NUMA
        binding) as the driver's own reference run, so the two numbers agree."""
        cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--config',
               config, '--steps', '200', '--warmup', '3', '--ref-seconds', str(budget_s),
               '--batch', str(self.B)]
        if config == 'clevr':
            cmd += ['--layouts', self.layouts]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
            line = json.loads(r.stdout.strip().splitlines()[-1])
            cb = line['cpu_baseline']
            cb['value'] = line['value']
            cb['median_ms_per_step'] = line.get('median_ms_per_step')
            return cb
        except Exception as e:
            return {'error': repr(e)}

    def close(self):
        self.pool = None
        self.ex = None
        self.feats = self.wvs = self.outs = None
        self.torch.cuda.empty_cache()


def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from n2nmn_b200 import synth
    from n2nmn_b200.executor import LayoutExecutor

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device. The product path has no CPU fallback.')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = bind_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    wl = WORKLOADS[args.config]
    B = args.batch or wl['B']
    layouts = args.layouts or wl['layouts']
    bn = Bench(torch, dist, args, wl, layouts, B, rank, world, dev, streams=args.streams or None,
               device_synth=(args.config not in ('clevr', 'shapes')))
    pool, ex, K = bn.pool, bn.ex, bn.K
    pk = peaks()

    # ---- headline: device-resident inputs, --warmup steps then exactly --steps timed steps
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    head = bn.headline(args.steps, args.warmup)
    launches = head['gpu_launches']
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name in ('scores', 'validity'):
            np.save(os.path.join(args.dump_outputs, name + '.npy'), head[name].astype(np.float32))

    # ---- the other two layout sets of SURVEY.md §8(d) (CLEVR: random valid; deep), same pool
    other_sets = None
    if args.config == 'clevr' and layouts == 'expert' and not args.no_other_sets:
        other_sets = {}
        for kind in ('random', 'deep'):
            otoks = [make_tokens(bn.asm, kind, B, wl['T'], seed=100 + 1000 * rank + i)
                     for i in range(8)]
            r = bn.timed(min(args.steps, 100), 12, 0.25, 1, toks=otoks)
            other_sets[kind] = {'value': r['value'], 'unit': UNIT, 'steps': r['timed_steps'],
                                'timed_region_s': r['timed_region_s'], 'nodes_per_batch': int(
                                    np.mean([int((t != bn.asm.EOS_idx).sum()) for t in otoks]))}

    # ---- e2e: host (pinned) buffers in, host scores out, every step, through the public API
    e2e = None if args.no_e2e else bn.e2e(args.steps, 0.4)
    # secondary: the same with an fp16 feature store on the host (half the PCIe bytes)
    e2e_f16 = None if (args.no_e2e or args.config != 'clevr') else bn.e2e(args.steps, 0.4, True)

    # ---- strong scaling point (SURVEY.md §8d(i)): the SAME global batch split over the ranks
    strong = None
    if world > 1 and B % world == 0 and args.config == 'clevr':
        Bs = B // world
        sb = Bench(torch, dist, args, wl, layouts, Bs, rank, world, dev,
                   streams=args.streams or None)
        r = sb.timed(args.steps, args.warmup, 0.3, 1)
        strong = {'value': r['value'], 'unit': UNIT, 'global_batch': B, 'batch_per_gpu': Bs,
                  'ms_per_step': r['ms_per_step'], 'timed_region_s': r['timed_region_s'],
                  'scaling': 'strong'}
        sb.close()

    # ---- roofline of the dominant kernel + HBM fractions of the two latency kernels (rank 0)
    roof = bn.roofline(pk) if rank == 0 else {}
    if rank == 0 and 'roofline' in roof:
        roof['roofline']['grid_ctas'] = pool.proj_ctas if pool.proj_ctas > 0 else 148

    # ---- config 3: policy-search train step (fwd + bwd + ONE NCCL all-reduce + clip + Adam),
    #      T=10 as in exp_clevr/train_clevr_rl_gt_layout.py; reported beside the eval headline
    train = None
    if args.config == 'clevr' and not args.no_train:
        from n2nmn_b200.trainer import ModuleNetTrainer
        T_TRAIN, C, P = 10, wl['C'], bn.P
        tr_ex = LayoutExecutor('clevr', bn.feats[0], bn.wvs[0][:T_TRAIN].contiguous(), C, bn.asm,
                               weights=bn.weights, max_batch=B, max_T=T_TRAIN)
        tr = ModuleNetTrainer(tr_ex)
        ttok = [np.ascontiguousarray(synth.expert_mix_tokens(bn.asm, B, T_TRAIN)[
            :, np.random.RandomState(7 + i).permutation(B)]) for i in range(P)]
        twv = [w[:T_TRAIN].contiguous() for w in bn.wvs]
        tlab = [np.random.RandomState(11 + i).randint(0, C, size=B) for i in range(P)]
        lsp = torch.full((B,), -2.0, device=dev)
        for i in range(5):
            tr.train_step(bn.feats[i % P], twv[i % P], ttok[i % P], tlab[i % P], log_seq_prob=lsp,
                          sync=False)
        k_tr = max(50, min(args.steps, 200))
        bn.barrier()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for i in range(k_tr):
            out = tr.train_step(bn.feats[i % P], twv[i % P], ttok[i % P], tlab[i % P],
                                log_seq_prob=lsp, sync=False)
        t1e.record()
        bn.barrier()
        tms = bn.allmax(t0e.elapsed_time(t1e))
        # per-kernel device times of the step (library profiling mode: CUDA events around every
        # launch group) and the roofline of the backward weight-gradient contraction
        tr_ex.set_profiling(True)
        acc = {}
        n_prof = 10
        for i in range(n_prof):
            tr.train_step(bn.feats[i % P], twv[i % P], ttok[i % P], tlab[i % P], log_seq_prob=lsp,
                          sync=False)
            torch.cuda.synchronize()
            for name, us in tr_ex.launch_times():
                acc[name] = acc.get(name, 0.0) + us / n_prof
        tr_ex.set_profiling(False)
        gflops = tr_ex.last_step_info().get('bwd_gemm_flops', 0)
        tf32_peak = pk['bf16_tflops'] / 2
        troof = None
        if gflops and acc.get('feat_grad_kernel'):
            tfs = gflops / (acc['feat_grad_kernel'] * 1e-6) / 1e12
            troof = {'kernel': 'wgrad_umma_kernel (dW = sum X^T B: tcgen05 kind::tf32, both operands '
                               'MN-major via TMA)',
                     'bound': 'tensor', 'achieved': tfs, 'peak': tf32_peak, 'unit': 'TFLOP/s',
                     'frac': tfs / tf32_peak, 'avg_launch_us': acc['feat_grad_kernel'],
                     'flops_per_launch': gflops,
                     'peak_source': pk['source'] + '; TF32 peak taken as bf16 burst / 2'}
        train = {'questions_per_sec': world * B * k_tr / (tms * 1e-3), 'kernel_us': acc,
                 'roofline': troof,
                 'ms_per_step': tms / k_tr, 'steps': k_tr, 'global_batch': B * world,
                 'T_decoder': T_TRAIN, 'last_avg_sample_loss': float(out['avg_sample_loss']),
                 'what': 'fwd + bwd + all-reduce(flat grads, %d floats) + per-tensor clip + Adam '
                         '+ weight re-pack' % (tr.flat_size + 1)}
        del tr, tr_ex

    # ---- (f1) the layout generator that feeds the path: one batch of 64 questions through the
    #      attentional seq2seq at the CLEVR sizes (exp_clevr/train_clevr_*.py), greedy decoding
    layout_gen = None
    if rank == 0 and world == 1 and args.config == 'clevr' and not args.no_seq2seq:
        layout_gen = seq2seq_measure(torch, bn.asm, dev, B)

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = bn.cpu_baseline(args.cpu_seconds, args.config)

    info = ex.last_step_info()
    pool_cfg = {'streams': K, 'host_threads': K, 'tree_cluster_ctas': pool.tree_cluster,
                'proj_grid_ctas': pool.proj_ctas if pool.proj_ctas > 0 else 148}

    # ---- the other BASELINE.json workloads at their real sizes (N=1 only): q/s, roofline, CPU port
    others = None
    if world == 1 and args.config == 'clevr' and layouts == 'expert' and not args.no_other_configs:
        others = {}
        bn.close()
        for name in ('shapes', 'vqa514', 'vqa2050', 'stress'):
            w2 = WORKLOADS[name]
            try:
                ob = Bench(torch, dist, args, w2, w2['layouts'], w2['B'], rank, world, dev,
                           streams=4, device_synth=(name != 'shapes'))
                r = ob.timed(min(args.steps, 40), 8, 0.3, 1)
                entry = {'workload': workload_title(w2, w2['layouts']), 'value': r['value'],
                         'unit': UNIT, 'ms_per_step': r['ms_per_step'],
                         'timed_region_s': r['timed_region_s'], 'repeats': r['repeats'],
                         'streams': ob.K, 'resident_batches': ob.P,
                         'cache': cache_note(ob)}
                entry.update(ob.roofline(pk))
                oi = ob.ex.last_step_info()
                entry['nodes_per_batch'] = oi['num_nodes']
                entry['max_depth'] = oi['max_depth']
                if not args.no_cpu_baseline:
                    entry['cpu_baseline'] = ob.cpu_baseline(3.0, name)
                others[name] = entry
                ob.close()
                del ob
            except Exception as e:   # one workload failing must not lose the headline line
                others[name] = {'error': repr(e)}

    if rank == 0:
        line = {
            'metric': wl['metric'], 'value': head['value'], 'unit': UNIT, 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': head['ms_per_step'],
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'tf32 (fp32 in/out, fp32 accumulate)', 'data': 'synthetic',
            'timed_steps': head['timed_steps'], 'timed_region_s': head['timed_region_s'],
            'config': dict({'workload': workload_title(wl, layouts), 'global_batch': B * world,
                            'parallelism': 'dp%d (question shards, no collective)' % world,
                            'cache': cache_note(bn),
                            'executor': 'wave' if args.wave else 'tree',
                            'nodes_per_batch': info['num_nodes'], 'max_depth': info['max_depth']},
                           **pool_cfg),
            'clocks': clocks, 'e2e': e2e, 'e2e_f16_host_features': e2e_f16,
            'gpu_launches': int(launches),
            'host_enqueue_ms_per_step': head['host_enqueue_ms_per_step'], 'host_numa': numa,
            'roofline': roof.get('roofline'), 'roofline_text': roof.get('roofline_text'),
            'roofline_tree': roof.get('roofline_tree'), 'roofline_pool': roof.get('roofline_pool'),
            'kernel_us': roof.get('kernel_us'),
            'cpu_baseline': cpu, 'train_step': train, 'layout_generator': layout_gen,
            'other_layout_sets': other_sets,
            'strong_scaling': strong, 'other_configs': others,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cache_note(b):
    tot = b.P * b.batch_bytes / 1e6
    return 'inputs larger than L2: %d distinct resident batches (%.0f MB) walked round-robin' % (
        b.P, tot)


if __name__ == '__main__':
    main()
