#!/usr/bin/env python
"""Benchmark of the Tacotron-2 training hot path (forward + loss + backward) -- driver contract.

    python bench.py --gpus 1 --steps 5 --warmup 3                    # this framework, 1 GPU
    torchrun --nproc-per-node N ... bench.py --gpus N ...             # data parallel, one rank per GPU, NCCL all-reduce
    python bench.py --impl reference --steps 2 --warmup 1             # CPU reference arm (unmodified reference from oracle/_ref, host cores)

A "step" is one training step of the named configuration on one synthetic batch per GPU: embedding -> encoder ->
fused decoder -> postnet -> TacotronLoss -> backward (-> gradient all-reduce when N > 1).  Optimizer, data loading
and logging are excluded (SURVEY.md section 8d).  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'mel-frames/sec (train fwd+bwd)'
UNIT = 'mel-frames/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='generated_training')
    ap.add_argument('--batch', type=int, default=0, help='per-GPU batch (default: 60 for grouped encoders, 64 otherwise)')
    ap.add_argument('--text-len', type=int, default=180)
    ap.add_argument('--frames', type=int, default=900)
    ap.add_argument('--regularization', default='zoneout', choices=['zoneout', 'dropout'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--ref-frames', type=int, default=100,
                    help='frames per utterance of the CPU reference sample (reference arm / cpu_baseline): the first N of --frames')
    ap.add_argument('--no-extra-baselines', action='store_true',
                    help='skip the cfg-1 CPU timing and the eager-PyTorch-on-B200 timing of the unmodified reference (N=1 only)')
    ap.add_argument('--no-graph', action='store_true', help='issue every step from Python instead of replaying the captured CUDA graph')
    ap.add_argument('--breakdown', default='', help='write a per-kernel device-time table of one extra (untimed) step to this file')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32'],
                    help="bf16: tensor-core operands, fp32 master/state (BASELINE configs[1]); fp32: exact parity mode")
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='after the timed steps, write what the last timed step returned (the loss and every parameter gradient) as DIR/<name>.npy')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    return a


def workload(a):
    from multilingual_text_to_speech_b200 import configs
    hp = configs.apply(a.config, decoder_regularization=a.regularization)
    G = max(hp.language_number, 1)
    grouped = hp.encoder_type in ('generated', 'convolutional')
    B = a.batch or (60 if grouped else 64)      # 64 is not divisible by the 10 / 5 languages of the grouped encoders (SURVEY D6)
    if grouped and B % G:
        raise SystemExit(f'batch {B} must be divisible by the {G} languages of the grouped encoder')
    return hp, B, a.text_len, a.frames


def synth_batch(hp, B, L, T, seed, device, pin=False):
    """Synthetic batch of SURVEY section 8d: random symbols, randn mels, full lengths, language b % G, stop ones on the last frames."""
    import torch
    g = torch.Generator().manual_seed(seed)
    G = max(hp.language_number, 1)
    batch = {
        'text': torch.randint(1, hp.symbols_count() + 3, (B, L), generator=g),
        'text_length': torch.full((B,), L, dtype=torch.long),
        'target': torch.randn(B, hp.num_mels, T, generator=g),
        'target_length': torch.full((B,), T, dtype=torch.long),
        'stop_target': torch.zeros(B, T),
    }
    batch['stop_target'][:, T - hp.stop_frames:] = 1.0
    if hp.multi_speaker:
        batch['speakers'] = torch.randint(0, hp.speaker_number, (B,), generator=g)
    if hp.multi_language:
        batch['languages'] = torch.arange(B) % G
    if pin:
        batch = {k: v.pin_memory() for k, v in batch.items()}
    if device is not None:
        batch = {k: v.to(device) for k, v in batch.items()}
    return batch


# --------------------------------------------------------------------------------------------------
# roofline bookkeeping (SURVEY.md section 8d formula: naive algorithmic bytes of one decoder step, forward)
# --------------------------------------------------------------------------------------------------
def step_elements(B, L, M, D=1024, P=256, A=128, C=32, K=31, N=80):
    """SURVEY.md section 8d, ELEMENTS touched by one decoder step (forward, whole batch, naive formulation), split by the persistent
    loop that owns them: (weights, activations) of the attention loop (attention-LSTM + location-sensitive attention) and of the
    generator loop (generator LSTM + frame / stop projections).  Their sum is W_step / ACT_step of the survey."""
    w_att = (4 * D * (P + M) + 4 * D * D + 8 * D) + (A * D + A * C + C * K + 2 * A)
    a_att = B * ((L * A + L * M + 2 * L + P + 2 * D) + (2 * D + 2 * L))
    w_gen = (4 * D * (D + M) + 4 * D * D + 8 * D) + (N * (D + M) + N + (D + M) + 1)
    a_gen = B * (2 * D + (2 * D + N + 1))
    return {'att': (w_att, a_att), 'gen': (w_gen, a_gen)}


def bytes_fwd_step(B, L, M, D=1024, P=256, A=128, C=32, K=31, N=80, w=4, a=4, part=None):
    el = step_elements(B, L, M, D, P, A, C, K, N)
    parts = [part] if part else ['att', 'gen']
    return sum(w * el[p][0] + a * el[p][1] for p in parts)


# which share of the per-step bytes a timed kernel is responsible for, and how many forward-equivalents it is (SURVEY 8d convention:
# the backward pass counts as 2 x forward -- one pass for dX, one for dW)
KERNEL_SHARE = {'lstm_loop_tc_kernel<att>': ('att', 1), 'lstm_loop_tc_kernel<gen>': ('gen', 1),
                'att_bwd_loop_kernel': ('att', 2), 'lstm_bwd_loop_tc_kernel': ('gen', 2), 'lstm_bwd_loop_kernel': ('gen', 2)}


def roofline_entry(name, ms, T, dims, peak, precision, traffic=None, fwd_equiv=1, part=None, note=None):
    """Fractions of the measured HBM peak for `ms` of device time against T x (share of BYTES_fwd_step) x fwd_equiv, at three element
    widths: the run's own (`frac`: bf16 runs are judged against the bf16 column of SURVEY 8d, w = a = 2), bf16 weights + fp32
    activations (`frac_mixed`), and the fp32-naive figure (`frac_fp32_naive`)."""
    def alg(w, a):
        return fwd_equiv * T * bytes_fwd_step(*dims, w=w, a=a, part=part)
    sec = ms * 1e-3
    own = (2, 2) if precision == 'bf16' else (4, 4)
    e = {'kernel': name, 'bound': 'hbm', 'unit': 'GB/s', 'peak': peak, 'avg_launch_ms': ms,
         'algorithmic_bytes_per_launch': alg(*own), 'achieved': alg(*own) / sec / 1e9, 'frac': alg(*own) / sec / 1e9 / peak,
         'frac_mixed': alg(2, 4) / sec / 1e9 / peak if precision == 'bf16' else None,
         'frac_fp32_naive': alg(4, 4) / sec / 1e9 / peak, 'traffic': traffic,
         'element_width': 'w=a=2 B (bf16 column of SURVEY 8d)' if precision == 'bf16' else 'w=a=4 B (fp32)',
         'algorithmic_bytes_formula': f'{fwd_equiv} x T x BYTES_fwd_step' + (f'[{part} loop share]' if part else '') + ' (SURVEY 8d)'}
    if note:
        e['note'] = note
    return e


def ncu_traffic(B, L, T):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the loop kernels from the committed ncu capture of the
    CURRENT kernels at this shape (profiles/r2/ncu_traffic.json, written by tools/ncu_traffic.py from the raw capture); {} if none."""
    path = os.path.join(ROOT, 'profiles', 'r2', 'ncu_traffic.json')
    if not os.path.exists(path):
        return {}
    d = json.load(open(path))
    if (d.get('B'), d.get('L'), d.get('T')) != (B, L, T):
        return {}
    return {k: v['dram_read'] + v['dram_write'] for k, v in d.get('kernels', {}).items()}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


DUMP_SAMPLE = 1 << 16      # elements kept of a larger gradient: the 152 gradients of the largest configuration stay below 64 MB


def dump_outputs(directory, model, loss):
    """What a training step hands its caller: the loss and every parameter's gradient, written as DIR/loss.npy and DIR/grad.<parameter
    name>.npy in float32.  A gradient of more than DUMP_SAMPLE elements is stored at DUMP_SAMPLE fixed positions of its flattened
    values (seeded, so the same for every run and every build), which lets two builds be compared output for output."""
    import numpy as np
    import torch
    arrays = {'loss': loss.detach().float().cpu().numpy()}
    for name, p in model.named_parameters():
        g = p.grad.detach()
        if g.numel() > DUMP_SAMPLE:
            idx = torch.randperm(g.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            g = g.flatten()[idx.to(g.device)]
        arrays['grad.' + name] = g.float().cpu().numpy()
    total = sum(v.nbytes for v in arrays.values())
    if total > 64 << 20:
        raise SystemExit(f'--dump-outputs: {total} bytes exceed the 64 MB bound')
    os.makedirs(directory, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(directory, name + '.npy'), v)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace('.', '').isdigit()]
        if not sm:
            return None
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith('active')})
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': float(self.rows[0][1]), 'reasons': reasons, 'samples': len(sm)}


# --------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port on the host cores
# --------------------------------------------------------------------------------------------------
def cpu_oracle_frames_per_s(a, steps, warmup, sample_frames=24):
    import torch
    from multilingual_text_to_speech_b200 import configs
    from multilingual_text_to_speech_b200.modules.tacotron2 import Tacotron
    from oracle import tacotron_oracle as O
    hp, B, L, _ = workload(a)
    T = sample_frames
    # torch's intra-op pool on a many-core host is dominated by fork/join overhead for this op mix (measured on the
    # 128-core B200 host: 12.6 frames/s with 128 threads); 16 threads is the best setting we found, and is what is reported.
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = Tacotron()                       # parameter container only (construction needs no GPU)
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
    for k in list(sd):
        if k.startswith('_decoder._prenet.') or k.startswith('_decoder._attention.'):
            sd[k] = sd[k[len('_decoder.'):]]
    ns = configs.as_namespace()
    b = synth_batch(hp, B, L, T, 1234, None)
    g = torch.Generator().manual_seed(7)
    D, P = hp.decoder_dimension, hp.prenet_dimension
    keep = lambda shape, p: (torch.rand(*shape, generator=g) >= p).float()   # noqa: E731
    tape = {'teacher': torch.ones(T, dtype=torch.bool), 'prenet0': keep((B, T + 1, P), 0.5), 'prenet1': keep((B, T + 1, P), 0.5),
            'att_h': keep((T, B, D), 0.1), 'gen_h': keep((T, B, D), 0.1), 'att_c': keep((T, B, D), 0.1), 'gen_c': keep((T, B, D), 0.1)}
    times = []
    for it in range(warmup + steps):
        for v in sd.values():
            if v.is_floating_point():
                v.grad = None
        t0 = time.perf_counter()
        post, pre, stop, align, spk, enc = O.tacotron_forward(sd, ns, b['text'], b['text_length'], b['target'], b['target_length'],
                                                              b.get('speakers'), b.get('languages'), tape, training=True)
        loss, _ = O.tacotron_loss(ns, hp.guided_attention_toleration, b['text_length'], b['target_length'], pre, b['target'], post,
                                  b['target'], stop, b['stop_target'], align, b.get('speakers'), spk)
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    med = statistics.median(times)
    sample = f'oracle port (torch CPU fp32), {a.config} B={B} L={L}, first {T} of {a.frames} frames, fwd+loss+bwd, {steps} timed steps'
    return B * T / med, med, cores, sample


def config_dict(a, world, B, L, T):
    """`config` of the JSON line: the same for this framework's arm and the reference arm."""
    return {'workload': f'{a.config} train fwd+bwd, B={B}/GPU L={L} T={T} ({a.regularization} cells), tf=1.0',
            'global_batch': world * B, 'parallelism': f'dp{world}',
            'precision': 'bf16 tensor-core operands, fp32 accumulate / master weights / states' if a.precision == 'bf16' else 'fp32',
            'l2': 'per-step working set (~5 GB of activations) >> 126 MB L2, no flush needed',
            'note': 'batch 64 is invalid for the 10-language grouped encoder (B % G == 0); shipped batch 60 used'}


def reference_cpu(a, steps, warmup):
    """The reference's own CPU implementation of the path on the host cores, on a BOUNDED sample of the workload: the same batch
    size / text length, but only the first `--ref-frames` of the T frames per utterance (a full T = 900 step of B = 60 takes ~1 min).
    oracle/_ref (the unmodified reference) when installed, else the oracle port."""
    hp, B, L, T = workload(a)
    Ts = min(a.ref_frames, T)
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    import reference_runner as R
    if R.available():
        r = R.time_cpu(a.config, a.regularization, B, L, Ts, steps, warmup)
        # second point at half the frames -> fixed (encoder, per-call) and per-frame cost -> what the full-T step would run at; the
        # truncated sample UNDER-states the reference by the share of the fixed cost (reported, never used as `value`)
        extra = None
        if Ts >= 20:
            r2 = R.time_cpu(a.config, a.regularization, B, L, Ts // 2, 1, 1, threads=r['cores'])
            per_frame = (r['s_per_step'] - r2['s_per_step']) / (Ts - Ts // 2)
            fixed = r['s_per_step'] - per_frame * Ts
            if per_frame > 0:
                extra = {'second_sample_frames': Ts // 2, 'second_sample_s_per_step': r2['s_per_step'], 'fixed_s': fixed,
                         's_per_frame_step': per_frame, 'extrapolated_full_T_frames_per_s': B * T / (fixed + per_frame * T)}
        sample = (f'UNMODIFIED reference (oracle/_ref: Tacotron.forward + TacotronLoss + backward, torch {_torch_version()} CPU fp32), '
                  f'{a.config} B={B} L={L}, first {Ts} of T={T} frames per utterance, {steps} timed step(s), threads scanned {r["thread_scan"]}')
        return {'value': r['frames_per_s'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'reference', 'sample': sample,
                'host_cores': os.cpu_count(), 'sample_frames': Ts, 'extrapolation': extra}, r['s_per_step']
    fps, med, cores, sample = cpu_oracle_frames_per_s(a, steps, warmup, sample_frames=min(Ts, 24))
    return {'value': fps, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample + ' (oracle/_ref not installed)',
            'host_cores': os.cpu_count(), 'sample_frames': min(Ts, 24)}, med


def _torch_version():
    import torch
    return torch.__version__


def run_reference(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    base, med = reference_cpu(a, a.steps, a.warmup)
    hp, B, L, T = workload(a)
    cfg = dict(config_dict(a, 1, B, L, T), precision='fp32 (reference arm: CPU)')
    cfg['workload'] += f' -- reference arm: bounded sample, first {base["sample_frames"]} of the T={T} frames per utterance'
    cfg['reference_sample_frames'] = base['sample_frames']
    line = {'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': med * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': cfg, 'cpu_baseline': base,
            'e2e': {'value': base['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def extra_baselines(a, threads):
    """BASELINE.md section 3: the mandated cfg-1 CPU timing (default Params = LJ Speech, B = 16, L = 180, T = 900, full length) and the
    unmodified reference in eager PyTorch on the B200 (the competitor on the same box) at this run's own workload."""
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    import reference_runner as R
    if not R.available():
        return {'unavailable': 'oracle/_ref not installed'}
    out = {}
    hp, B, L, T = workload(a)
    try:
        r = R.time_cpu('ljspeech', 'dropout', 16, 180, 900, 1, 1, threads=threads)
        out['cpu_cfg1_ljspeech_B16'] = {'value': r['frames_per_s'], 'unit': UNIT, 'cores': r['cores'], 's_per_step': r['s_per_step'],
                                        'sample': 'unmodified reference, default Params (LJ Speech), B=16 L=180 T=900 (full), fwd+loss+bwd, 1 warm-up + 1 timed step'}
    except Exception as exc:      # noqa: BLE001 -- a baseline must never take the bench line down
        out['cpu_cfg1_ljspeech_B16'] = {'error': repr(exc)[:200]}
    try:
        r = R.time_gpu_eager(a.config, a.regularization, B, L, T, steps=1, warmup=1)
        out['eager_pytorch_b200'] = {'value': r['frames_per_s'], 'unit': UNIT, 's_per_step': r['s_per_step'],
                                     'sample': f'unmodified reference, eager PyTorch fp32 (ATen / cuDNN / cuBLAS) on cuda:0, {a.config} B={B} L={L} T={T} (full), '
                                               'fwd+loss+bwd, 1 warm-up + 1 timed step'}
    except Exception as exc:      # noqa: BLE001
        out['eager_pytorch_b200'] = {'error': repr(exc)[:200]}
    return out


# --------------------------------------------------------------------------------------------------
# this framework
# --------------------------------------------------------------------------------------------------
def run_b200(a):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    entry.build()
    from multilingual_text_to_speech_b200 import _lib, functional as F
    from multilingual_text_to_speech_b200.modules.tacotron2 import Tacotron, TacotronLoss
    from multilingual_text_to_speech_b200.rng import MaskSource
    from multilingual_text_to_speech_b200.distributed import GradBucket

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl b200 needs a CUDA device: the hot path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    hp, B, L, T = workload(a)
    _lib.set_precision(a.precision)
    torch.manual_seed(0)
    model = Tacotron().to(dev).train()
    crit = TacotronLoss(hp.guided_attention_steps, hp.guided_attention_toleration, hp.guided_attention_gain)
    bucket = GradBucket(model, world)
    MaskSource.manual_seed(1234 + rank)
    host = synth_batch(hp, B, L, T, 1234 + rank, None, pin=True)
    resident = {k: v.to(dev) for k, v in host.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())
    F.PROFILE.clear()

    def eager_step(batch):
        bucket.zero()
        post, pre, stop, align, spk, enc = model(batch['text'], batch['text_length'], batch['target'], batch['target_length'],
                                                 batch.get('speakers'), batch.get('languages'), hp.teacher_forcing)
        loss, _ = crit(batch['text_length'], batch['target_length'], pre, batch['target'], post, batch['target'], stop,
                       batch['stop_target'], align, batch.get('speakers'), spk, enc, None)
        loss.backward()
        bucket.allreduce()
        return loss

    # the public way to run a step of fixed shape: forward + loss + backward captured ONCE into a CUDA graph and replayed
    # (multilingual_text_to_speech_b200.graph.GraphedTrainStep); the gradient all-reduce follows the replay
    graphed, launches_per_step, launch_mode = None, None, 'eager (one Python-issued launch sequence per step)'
    if not a.no_graph:
        try:
            from multilingual_text_to_speech_b200.graph import GraphedTrainStep
            n_before = _lib.launch_count()
            graphed = GraphedTrainStep(model, crit, bucket, resident, teacher_forcing=hp.teacher_forcing, warmup=max(a.warmup, 3))
            launches_per_step = (_lib.launch_count() - n_before) // (max(a.warmup, 3) + 1)
            launch_mode = 'CUDA graph replay of the captured step (GraphedTrainStep), gradient all-reduce after the replay'
        except Exception as exc:      # noqa: BLE001 -- capture is an optimisation; the eager path is the same kernels
            graphed, launch_mode = None, f'eager (graph capture failed: {exc!r})'[:300]
            torch.cuda.synchronize()

    def step(batch):
        if graphed is None:
            return eager_step(batch)
        loss = graphed(batch)
        bucket.allreduce()
        return loss

    def timed(n, from_host):
        """n steps bracketed by barrier + synchronize; device time by CUDA events; returns (max-over-ranks ms, last loss read on the host
        (from_host only), last loss tensor)."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss_val, loss = None, None
        for _ in range(n):
            if from_host and graphed is not None:
                batch = host                       # GraphedTrainStep copies the pinned host tensors into its static device buffers
            else:
                batch = {k: v.to(dev, non_blocking=True) for k, v in host.items()} if from_host else resident
            loss = step(batch)
            if from_host:
                loss_val = float(loss.detach())   # device -> host read of the step's result
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), loss_val, loss

    # the clock sampler (an nvidia-smi child process) starts BEFORE the warm-up: its NVML initialisation briefly contends with
    # the CUDA driver, which must not land inside the timed region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(a.warmup, 3)):
        step(resident)
    F.PROFILE.clear()
    n0 = _lib.launch_count()
    ncu_range = bool(os.environ.get('B200TTS_NCU_RANGE'))   # `ncu --profile-from-start off`: capture exactly the timed steps
    if graphed is None:
        F.PROFILE['enabled'] = True
        _lib.kernel_timing(True)          # CUDA events on the launching stream around the dominant kernels, inside the timed steps
    if ncu_range:
        torch.cuda.profiler.start()
    ms, _, last_loss = timed(a.steps, from_host=False)
    if ncu_range:
        torch.cuda.profiler.stop()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, model, last_loss)   # before the steps below overwrite the gradients
    launches = (_lib.launch_count() - n0) if graphed is None else launches_per_step * a.steps
    if graphed is not None:
        # events cannot be timed inside a replayed graph: the per-kernel durations come from the SAME kernels issued eagerly, a.steps
        # steps on the same inputs right after the timed replays (the kernels are launch-order independent; only the gaps differ)
        F.PROFILE['enabled'] = True
        _lib.kernel_timing(True)
        for _ in range(a.steps):
            eager_step(resident)
    F.PROFILE['enabled'] = False
    torch.cuda.synchronize()
    ktimes = _lib.kernel_timing_read()    # {kernel: (total ms, launches)} over a.steps steps
    _lib.kernel_timing(False)
    dec_ms = [s.elapsed_time(e) for s, e in F.PROFILE.get('decoder_fwd', [])]
    decb_ms = [s.elapsed_time(e) for s, e in F.PROFILE.get('decoder_bwd', [])]
    ms_e2e, loss_val, _ = timed(a.steps, from_host=True)
    clocks = sampler.stop() if rank == 0 else None
    if a.breakdown and rank == 0:       # CUPTI kernel times of ONE extra step (not part of any reported number)
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eager_step(resident)
            torch.cuda.synchronize()
        import collections
        import tempfile
        trace = os.path.join(tempfile.gettempdir(), f'b200tts_trace_{os.getpid()}.json')
        prof.export_chrome_trace(trace)
        agg = collections.defaultdict(lambda: [0, 0.0])
        for ev in json.load(open(trace)).get('traceEvents', []):
            if ev.get('cat') in ('kernel', 'gpu_memcpy', 'gpu_memset') and 'dur' in ev:
                name = ev['name'].replace('b200tts::(anonymous namespace)::', '').replace('void ', '').split('(')[0][:56]
                key = (name, str(ev.get('args', {}).get('grid', '')))
                agg[key][0] += 1
                agg[key][1] += float(ev['dur'])
        os.remove(trace)
        tot = sum(v[1] for v in agg.values())
        with open(a.breakdown, 'w') as f:
            f.write(f'{"kernel":58s} {"grid":18s} {"n":>5s} {"total_us":>11s} {"avg_us":>10s} {"share":>7s}\n')
            for (name, grid), v in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                f.write(f'{name:58s} {grid:18s} {v[0]:5d} {v[1]:11.1f} {v[1] / v[0]:10.2f} {100 * v[1] / max(tot, 1e-9):6.1f}%\n')
            f.write(f'{"TOTAL":58s} {"":18s} {sum(v[0] for v in agg.values()):5d} {tot:11.1f}\n')
    if rank == 0:
        frames = world * B * T * a.steps
        value = frames / (ms * 1e-3)
        M = hp.encoder_dimension + (hp.speaker_embedding_dimension if hp.multi_speaker else 0) + \
            (hp.language_embedding_dimension if hp.multi_language else 0)
        peak, peak_src = measured_peaks()
        dims = (B, L, M, hp.decoder_dimension, hp.prenet_dimension, hp.attention_dimension, hp.attention_location_dimension,
                hp.attention_kernel_size, hp.num_mels)
        traffic = ncu_traffic(B, L, T)
        roofs = []
        for kname, (tot, cnt) in ktimes.items():
            if kname in KERNEL_SHARE and cnt:
                part, eq = KERNEL_SHARE[kname]
                roofs.append(roofline_entry(kname, tot / cnt, T, dims, peak, a.precision, traffic.get(kname), eq, part))
        if dec_ms:
            roofs.append(roofline_entry('decoder forward op (both forward loops + the time-batched GEMMs around them)', statistics.mean(dec_ms),
                                        T, dims, peak, a.precision, None, 1, None))
        if decb_ms:
            roofs.append(roofline_entry('decoder backward op (both reverse loops, post pass, dW / dX GEMMs)', statistics.mean(decb_ms),
                                        T, dims, peak, a.precision, None, 2, None))
        roofs.append(roofline_entry('whole training step (encoder, decoder, postnet, loss, backward)', ms / a.steps, T, dims, peak, a.precision,
                                    None, 3, None, note='3 x T x BYTES_fwd_step: decoder bytes only, the encoder / postnet / loss time counts against them'))
        loops = [r for r in roofs if r['kernel'] in KERNEL_SHARE]
        roof = dict(max(loops, key=lambda r: r['avg_launch_ms'])) if loops else (dict(roofs[0]) if roofs else None)
        if roof:
            roof['peak_source'] = peak_src
            roof['why_this_kernel'] = 'largest device time among the kernels of the step (CUDA events around each launch inside the timed steps)'
            roof['timing'] = {k: {'ms_per_launch': v[0] / max(v[1], 1), 'launches': v[1]} for k, v in ktimes.items()}
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': max(a.warmup, 3),
                'ms_per_step': ms / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16' if a.precision == 'bf16' else 'f32', 'data': 'synthetic',
                'config': dict(config_dict(a, world, B, L, T), launch=launch_mode),
                'clocks': clocks, 'gpu_launches': int(launches),
                'e2e': {'value': frames / (ms_e2e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': int(h2d_bytes), 'd2h_bytes_per_step': 4,
                        'loss': loss_val},
                'roofline': roof, 'rooflines': roofs}
        if world == 1 and not a.no_cpu_baseline:
            line['cpu_baseline'], _ = reference_cpu(a, 1, 0)
            if not a.no_extra_baselines:
                line['baselines'] = extra_baselines(a, line['cpu_baseline']['cores'])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_b200(a)


if __name__ == '__main__':
    main()
