"""CPU checks of bench.py: the reference arm (the unmodified reference from oracle/_ref when installed, else the oracle port, on the
host cores) prints one well-formed JSON line, and the roofline bookkeeping reproduces the SURVEY section 8d figures."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bytes_fwd_step_matches_survey_table():
    sys.path.insert(0, ROOT)
    import bench
    # SURVEY 8d: cfg 2 (B = 64, L = 180, M = 288) -> 86.54 MB per forward step in fp32; cfg 1 (B = 16, M = 512) -> 80.38 MB
    assert abs(bench.bytes_fwd_step(64, 180, 288) / 1e6 - 86.54) < 0.01
    assert abs(bench.bytes_fwd_step(16, 180, 512) / 1e6 - 80.38) < 0.01
    # bf16 column (w = a = 2) and the split by persistent loop
    assert abs(bench.bytes_fwd_step(64, 180, 288, w=2, a=2) / 1e6 - 43.27) < 0.01
    both = bench.bytes_fwd_step(60, 180, 288, w=2, a=2)
    assert bench.bytes_fwd_step(60, 180, 288, w=2, a=2, part='att') + bench.bytes_fwd_step(60, 180, 288, w=2, a=2, part='gen') == both
    # the judge's round-1 recomputation: 42.6 MB per step at B = 60 in bf16; 20.62 ms for T = 900 steps against 6575 GB/s -> 0.283
    e = bench.roofline_entry('x', 20.62, 900, (60, 180, 288), 6575.1, 'bf16')
    assert abs(both / 1e6 - 42.6) < 0.05 and abs(e['frac'] - 0.283) < 0.002 and abs(e['frac_fp32_naive'] - 0.5655) < 0.002


def test_dump_outputs_writes_loss_and_gradients(tmp_path):
    """--dump-outputs: the loss and one float32 array per parameter gradient; a gradient above DUMP_SAMPLE elements is kept at the
    same seeded positions on every call."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(300, 300), torch.nn.Linear(300, 2))
    loss = model(torch.randn(4, 300)).square().mean()
    loss.backward()
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), model, loss)
    names = sorted(p.name for p in (tmp_path / 'a').iterdir())
    assert names == ['grad.0.bias.npy', 'grad.0.weight.npy', 'grad.1.bias.npy', 'grad.1.weight.npy', 'loss.npy']
    for n in names:
        a, b = np.load(tmp_path / 'a' / n), np.load(tmp_path / 'b' / n)
        assert a.dtype == np.float32 and np.array_equal(a, b), n
    assert float(np.load(tmp_path / 'a' / 'loss.npy')) == float(loss.detach())
    assert np.array_equal(np.load(tmp_path / 'a' / 'grad.1.weight.npy'), model[1].weight.grad.numpy())
    big = np.load(tmp_path / 'a' / 'grad.0.weight.npy')
    assert big.shape == (bench.DUMP_SAMPLE,) and set(big.tolist()) <= set(model[0].weight.grad.flatten().tolist())


def test_reference_arm_prints_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS='4')
    res = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                          '--frames', '900', '--ref-frames', '12', '--batch', '10', '--text-len', '40'], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'dtype', 'data',
                'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    installed = os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'modules', 'tacotron2.py'))
    assert line['impl'] == 'reference' and line['value'] > 0 and line['cpu_baseline']['kind'] == ('reference' if installed else 'port')
    # the bounded sample is named: the arm never claims the full T
    assert line['config']['reference_sample_frames'] == 12 and 'first 12 of the T=900' in line['config']['workload']
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
