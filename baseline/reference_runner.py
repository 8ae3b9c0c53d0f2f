"""Drive the UNMODIFIED reference (oracle/_ref/, installed by oracle/install_reference.py) through its own public API:
`Tacotron()` + `TacotronLoss` from modules/tacotron2.py, configured by its own params/*.json -- no code of this repository on that path.

Used by `bench.py --impl reference` (CPU, all host threads it can use) and by bench.py's extra baselines (the mandated cfg-1 CPU
timing, eager PyTorch on the B200).  Test / measurement infrastructure only: the product never imports this module.
"""
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.path.dirname(HERE), 'oracle', '_ref')


def available():
    return os.path.exists(os.path.join(REF, 'modules', 'tacotron2.py'))


_loaded = None


def load():
    """Import the reference (recipe of SURVEY appendix C: `import utils` before modules.tacotron2).  Returns (hp, Tacotron, TacotronLoss)."""
    global _loaded
    if _loaded is None:
        if not available():
            raise RuntimeError('oracle/_ref is not installed: run `python oracle/install_reference.py` where the original sources exist')
        sys.dont_write_bytecode = True
        if REF not in sys.path:
            sys.path.insert(0, REF)
        import utils  # noqa: F401
        from params.params import Params as hp
        from modules.tacotron2 import Tacotron, TacotronLoss
        _loaded = (hp, Tacotron, TacotronLoss, dict(hp.state_dict()))
    return _loaded[:3]


CONFIG_JSON = {'generated_training': 'generated_training.json', 'shared_switching': 'shared_switching.json',
               'generated_switching': 'generated_switching.json', 'ljspeech': None}


def configure(config, regularization, speakers=7):
    hp, Tacotron, TacotronLoss = load()
    hp.load_state_dict(_loaded[3])                      # defaults (JSON overlays are cumulative on the static class)
    if CONFIG_JSON[config]:
        hp.load(os.path.join(REF, 'params', CONFIG_JSON[config]))
    hp.decoder_regularization = regularization
    hp.language_number = len(hp.languages) if hp.multi_language else 0      # train.py:239-240
    hp.speaker_number = speakers if hp.multi_speaker else 0
    return hp


def synth_batch(hp, B, L, T, seed):
    """Same synthetic batch as bench.py's own arm (SURVEY section 8d)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    G = max(hp.language_number, 1)
    batch = {'text': torch.randint(1, hp.symbols_count() + 3, (B, L), generator=g),
             'text_length': torch.full((B,), L, dtype=torch.long),
             'target': torch.randn(B, hp.num_mels, T, generator=g),
             'target_length': torch.full((B,), T, dtype=torch.long),
             'stop_target': torch.zeros(B, T)}
    batch['stop_target'][:, T - hp.stop_frames:] = 1.0
    batch['speakers'] = torch.randint(0, hp.speaker_number, (B,), generator=g) if hp.multi_speaker else None
    batch['languages'] = (torch.arange(B) % G) if hp.multi_language else None
    return batch


class Runner:
    """One configured reference model + batch; `step()` = forward + TacotronLoss + backward (train.py:63-83)."""

    def __init__(self, config, regularization, B, L, T, device='cpu', seed=1234):
        import torch
        self.torch = torch
        self.hp = configure(config, regularization)
        _, Tacotron, TacotronLoss = load()
        torch.manual_seed(0)
        self.model = Tacotron().to(device).train()
        hp = self.hp
        self.crit = TacotronLoss(hp.guided_attention_steps, hp.guided_attention_toleration, hp.guided_attention_gain)
        self.device = device
        self.batch = {k: (v.to(device) if v is not None else None) for k, v in synth_batch(hp, B, L, T, seed).items()}
        if hp.encoder_type in ('simple', 'separate', 'shared'):
            # pack_padded_sequence wants its lengths on the CPU (modules/encoder.py:41 under a modern torch; SURVEY 8c)
            self.batch['text_length'] = self.batch['text_length'].cpu()
        self.frames = B * T

    def step(self):
        b, hp = self.batch, self.hp
        self.model.zero_grad(set_to_none=True)
        post, pre, stop, align, spk, enc = self.model(b['text'], b['text_length'], b['target'], b['target_length'], b['speakers'],
                                                      b['languages'], hp.teacher_forcing)
        classifier = self.model._reversal_classifier if hp.reversal_classifier else None
        loss, _ = self.crit(b['text_length'].to(stop.device), b['target_length'], pre, b['target'], post, b['target'], stop, b['stop_target'],
                            align, b['speakers'], spk, enc, classifier)
        loss.backward()
        return loss

    def timed_step(self):
        torch = self.torch
        if self.device != 'cpu':
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = self.step()
        if self.device != 'cpu':
            torch.cuda.synchronize()
        return time.perf_counter() - t0, float(loss.detach())


def pick_threads(runner, candidates, verbose=False):
    """One step per candidate thread count; the fastest is used for the timed steps (torch's intra-op pool does not scale to all cores
    of a 128-core host for this op mix: the fork / join overhead of ~10^5 tiny ops dominates)."""
    import torch
    best, best_t, seen = None, None, {}
    for n in candidates:
        torch.set_num_threads(n)
        dt, _ = runner.timed_step()
        seen[n] = dt
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best, seen


def time_cpu(config, regularization, B, L, T, steps, warmup, threads=None):
    """-> dict(frames_per_s, s_per_step, cores, thread_scan)."""
    import torch
    r = Runner(config, regularization, B, L, T, 'cpu')
    ncpu = os.cpu_count() or 1
    scan = None
    if threads is None:
        # measured on the 128-core B200 host: 8 -> 2.8 s, 16 -> 2.0 s, 32 -> 2.9 s, 64 -> 6.3 s, 128 -> 403 s per step (torch's intra-op
        # pool collapses on ~10^5 tiny ops); the scan therefore stops at 32 threads
        cands = sorted({n for n in (8, 16, 32) if n <= ncpu} or {ncpu})
        threads, scan = pick_threads(r, cands)          # the scan steps double as warm-up
        for _ in range(max(0, warmup - len(cands))):
            r.timed_step()
    else:
        torch.set_num_threads(threads)
        for _ in range(warmup):
            r.timed_step()
    times = [r.timed_step()[0] for _ in range(steps)]
    med = statistics.median(times)
    return {'frames_per_s': r.frames / med, 's_per_step': med, 'cores': threads, 'thread_scan': scan, 'frames': r.frames}


def time_gpu_eager(config, regularization, B, L, T, steps=1, warmup=1):
    """The same reference in eager PyTorch on cuda:0 (ATen / cuDNN / cuBLAS): the competitor on the same box (SURVEY 2.1)."""
    import torch
    r = Runner(config, regularization, B, L, T, 'cuda:0')
    for _ in range(warmup):
        r.timed_step()
    times = [r.timed_step()[0] for _ in range(steps)]
    med = statistics.median(times)
    del r
    torch.cuda.empty_cache()
    return {'frames_per_s': B * T / med, 's_per_step': med, 'frames': B * T}
