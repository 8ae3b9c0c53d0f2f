"""Shared test helpers: golden-fixture loading and comparison utilities."""
import os
import sys
import json
import types
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')

GOLDEN_CASES = ['lj_dropout', 'lj_zoneout', 'lj_mixed_tf', 'lj_eval_free', 'generated_training',
                'shared_switching', 'generated_switching']


class Golden:
    """One golden case produced by tests/golden/make_golden.py from the unmodified reference."""

    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN_DIR, name + '.npz'))
        self.name = name
        self.meta = json.loads(bytes(z['meta']).decode())
        self.hp = types.SimpleNamespace(**self.meta['hp'])
        self.B, self.L, self.T = self.meta['B'], self.meta['L'], self.meta['T']
        self.tf, self.train = self.meta['tf'], self.meta['train']
        self.losses = self.meta['losses']
        self.inputs, self.sd, self.sd_after, self.tape, self.out, self.grad = {}, {}, {}, {}, {}, {}
        for key in z.files:
            if key == 'meta':
                continue
            group, _, rest = key.partition('.')
            arr = torch.from_numpy(z[key])
            {'in': self.inputs, 'sd': self.sd, 'sd_after': self.sd_after, 'tape': self.tape,
             'out': self.out, 'grad': self.grad}[group][rest] = arr
        self.tape = {k: (v.bool() if k == 'teacher' else v.float()) for k, v in self.tape.items()}

    def cast_sd(self, dtype, requires_grad=False):
        sd = {}
        for k, v in self.sd.items():
            if v.is_floating_point():
                t = v.to(dtype).clone()
                t.requires_grad_(requires_grad)
                sd[k] = t
            else:
                sd[k] = v.clone()
        # shared modules: the reference registers prenet / attention twice (top level and under _decoder)
        for k in list(sd):
            if k.startswith('_decoder._prenet.') or k.startswith('_decoder._attention.'):
                sd[k] = sd[k[len('_decoder.'):]]
        return sd

    def tape_cast(self, dtype):
        return {k: (v if k == 'teacher' else v.to(dtype)) for k, v in self.tape.items()}


SAMPLE_MAX = 8192


def sample_index(numel):
    """Fixed, seeded flat positions at which a tensor larger than SAMPLE_MAX elements is stored in a golden file (None: stored whole)."""
    if numel <= SAMPLE_MAX:
        return None
    return torch.randperm(numel, generator=torch.Generator().manual_seed(0))[:SAMPLE_MAX].sort().values


def golden_array(t):
    """What a golden file stores of `t`: the tensor itself, or its values at sample_index(t.numel())."""
    t = t.detach().cpu()
    idx = sample_index(t.numel())
    return t if idx is None else t.flatten()[idx]


def digest(t):
    """float64 [sum, sum of squares, position-weighted sum]: pins a regenerated tensor (weights, inputs) to the one a fixture was made from."""
    v = t.detach().cpu().double().flatten()
    return torch.stack([v.sum(), (v * v).sum(), (v * torch.linspace(-1.0, 1.0, v.numel(), dtype=torch.float64)).sum()])


class ModuleGolden:
    """One case of tests/golden/modules_*.npz (tests/golden/make_golden_modules.py): arrays by name, as float64 torch tensors."""

    def __init__(self, file, case):
        z = np.load(os.path.join(GOLDEN_DIR, file + '.npz'))
        self.a = {k[len(case) + 1:]: torch.from_numpy(z[k]).double() for k in z.files if k.startswith(case + '.')}

    def __getitem__(self, name):
        return self.a[name]

    def check_digest(self, name, t):
        got, want = digest(t), self.a['digest.' + name]
        assert torch.allclose(got, want, rtol=1e-9, atol=1e-9), f'{name}: regenerated {got.tolist()} != fixture {want.tolist()}'

    def assert_close(self, actual, name, rtol, atol):
        """`actual` (whole tensor) against the stored (possibly sampled) reference values of `name`."""
        assert_close(golden_array(actual), self.a[name], rtol, atol, name)


def max_abs(a, b):
    return float((a.double() - b.double()).abs().max()) if a.numel() else 0.0


def assert_close(actual, expected, rtol=1e-3, atol=1e-4, what=''):
    actual, expected = actual.detach().double().cpu(), expected.detach().double().cpu()
    assert actual.shape == expected.shape, f'{what}: shape {tuple(actual.shape)} vs {tuple(expected.shape)}'
    diff = (actual - expected).abs()
    tol = atol + rtol * expected.abs()
    bad = diff > tol
    if bool(bad.any()):
        idx = int(torch.argmax((diff - tol).flatten()))
        raise AssertionError(f'{what}: {int(bad.sum())}/{bad.numel()} outside rtol={rtol} atol={atol}; '
                             f'max|diff|={float(diff.max()):.3e} at flat {idx}: '
                             f'{float(actual.flatten()[idx]):.6e} vs {float(expected.flatten()[idx]):.6e}')
