"""Golden vectors of single reference modules (CPU, fp32) for tests/test_gpu_modules.py; needs a checkout of the original project.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_modules.py <original project checkout>

Each case replays the seeded set-up of its test exactly (the reference module and this package's twin are constructed in the same
order, so both the weights and the inputs drawn after them are the ones the test regenerates), runs the UNMODIFIED reference module
forward + backward, and stores digests of the weights / inputs (so the test can prove it regenerated the same ones), the outputs and
all gradients.  Tensors larger than helpers.SAMPLE_MAX elements are stored at fixed seeded positions, with their max |value| whole.
  modules_lstm.npz        ZoneoutLSTMCell / DropoutLSTMCell, eval mode (modules/layers.py:18-47)
  modules_generated.npz   Conv1dGenerated + BatchNorm1dGenerated, train and eval mode (modules/generated.py:7-96)
  modules_attention.npz   LocationSensitiveAttention.reset + three steps (modules/attention.py)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def _store(out, case, name, t, absmax=False):
    from helpers import golden_array
    out[f'{case}.{name}'] = golden_array(t).numpy()
    if absmax:
        out[f'{case}.absmax.{name}'] = np.float64(t.detach().abs().max())


def _digest(out, case, name, t):
    from helpers import digest
    out[f'{case}.digest.{name}'] = digest(t).numpy()


def lstm_cases(out):
    import torch
    from modules.layers import ZoneoutLSTMCell as RZ, DropoutLSTMCell as RD
    from multilingual_text_to_speech_b200.modules.layers import ZoneoutLSTMCell, DropoutLSTMCell
    for kind in ('zoneout', 'dropout'):
        torch.manual_seed(3)
        I, H, B = 544, 1024, 7
        ref = (RZ(I, H, 0.1, 0.1) if kind == 'zoneout' else RD(I, H, 0.1)).eval()
        (ZoneoutLSTMCell(I, H, 0.1, 0.1) if kind == 'zoneout' else DropoutLSTMCell(I, H, 0.1))
        x, h, c = torch.randn(B, I), torch.randn(B, H), torch.randn(B, H)
        xr, hr, cr = (t.clone().requires_grad_(True) for t in (x, h, c))
        h1, c1 = ref(xr, hr, cr)
        gh, gc = torch.randn(B, H), torch.randn(B, H)
        ((h1 * gh).sum() + (c1 * gc).sum()).backward()
        for n, p in ref.named_parameters():
            _digest(out, kind, n, p)
            _store(out, kind, 'd' + n, p.grad, absmax=True)
        for n, t in (('x', x), ('h', h), ('c', c), ('gh', gh), ('gc', gc)):
            _digest(out, kind, n, t)
        for n, t in (('h', h1), ('c', c1), ('dx', xr.grad), ('dh', hr.grad), ('dc', cr.grad)):
            _store(out, kind, n, t)


def generated_cases(out):
    import torch
    from modules.generated import Conv1dGenerated as RC, BatchNorm1dGenerated as RB
    from multilingual_text_to_speech_b200.modules.generated import Conv1dGenerated, BatchNorm1dGenerated
    for train in (True, False):
        case = 'train' if train else 'eval'
        torch.manual_seed(5)
        G, gd, bn, Cin, Cout, k, dil, NB, L = 3, 6, 4, 8, 12, 3, 2, 4, 21
        e = torch.randn(G, gd)
        x = torch.randn(NB, G * Cin, L + (k - 1) * dil)
        rc = RC(gd, bn, G * Cin, G * Cout, k, padding=0, dilation=dil, groups=G, bias=False).train(train)
        Conv1dGenerated(gd, bn, G * Cin, G * Cout, k, padding=0, dilation=dil, groups=G, bias=False)
        rb = RB(gd, bn, G * Cout, groups=G).train(train)
        BatchNorm1dGenerated(gd, bn, G * Cout, groups=G)
        er, xr = e.clone().requires_grad_(True), x.clone().requires_grad_(True)
        y1 = rc(er, xr)
        z1 = rb(er, y1)
        gz = torch.randn_like(z1)
        (z1 * gz).sum().backward()
        params = [('conv.' + n, p) for n, p in rc.named_parameters()] + [('bn.' + n, p) for n, p in rb.named_parameters()]
        for n, p in params:
            _digest(out, case, n, p)
            _store(out, case, 'd' + n, p.grad, absmax=True)
        for n, t in (('e', e), ('x', x), ('gz', gz)):
            _digest(out, case, n, t)
        _store(out, case, 'y', y1)
        _store(out, case, 'z', z1)
        _store(out, case, 'de', er.grad, absmax=True)
        _store(out, case, 'dx', xr.grad, absmax=True)
        _store(out, case, 'running_mean', rb.running_mean)
        _store(out, case, 'running_var', rb.running_var)
        out[f'{case}.num_batches_tracked'] = np.float64(int(rb.num_batches_tracked))


def attention_case(out):
    import torch
    from modules.attention import LocationSensitiveAttention as RA
    from multilingual_text_to_speech_b200.modules.attention import LocationSensitiveAttention
    case = 'attention'
    torch.manual_seed(7)
    B, L, M, D, A, C, K = 5, 37, 288, 1024, 128, 32, 31
    ref = RA(K, C, False, A, D, M)
    LocationSensitiveAttention(K, C, False, A, D, M)
    with torch.no_grad():
        for prm in ref.parameters():
            prm.mul_(3.0)
    lens = torch.tensor([37, 30, 37, 12, 25])
    mask = torch.arange(L)[None, :] < lens[:, None]
    memory = torch.randn(B, L, M)
    queries = [torch.randn(B, D) for _ in range(3)]
    mr = memory.clone().requires_grad_(True)
    qr = [q.clone().requires_grad_(True) for q in queries]
    ref.reset(mr, B, L, memory.device)
    gen = torch.Generator().manual_seed(1)
    loss = 0.0
    for step in range(3):
        c1, w1 = ref(qr[step], mr, mask, None)
        _store(out, case, f'weights{step}', w1)
        _store(out, case, f'context{step}', c1)
        gc, gw = torch.randn(B, M, generator=gen), torch.randn(B, L, generator=gen)
        loss = loss + (c1 * gc).sum() + (w1 * gw).sum()
    loss.backward()
    for n, p in ref.named_parameters():
        _digest(out, case, n, p)
        _store(out, case, 'd' + n, p.grad, absmax=True)
    _digest(out, case, 'memory', memory)
    for step in range(3):
        _digest(out, case, f'query{step}', queries[step])
        _store(out, case, f'dquery{step}', qr[step].grad, absmax=True)
    _store(out, case, 'dmemory', mr.grad, absmax=True)


def main(ref_root):
    sys.path[:0] = [ref_root, ROOT, os.path.dirname(HERE)]
    import utils  # noqa: F401  (must precede the reference's modules: circular import in the reference)
    for name, fill in (('modules_lstm', lstm_cases), ('modules_generated', generated_cases), ('modules_attention', attention_case)):
        out = {}
        fill(out)
        path = os.path.join(HERE, name + '.npz')
        np.savez_compressed(path, **out)
        print(f'{name}: {len(out)} arrays, {os.path.getsize(path) / 1024:.0f} KiB')


if __name__ == '__main__':
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
