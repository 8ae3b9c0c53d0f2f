"""Module-level forwards of the boundary (SURVEY 8b) against the UNMODIFIED reference classes (CPU, fp32):
ZoneoutLSTMCell / DropoutLSTMCell (modules/layers.py:18-47), Conv1dGenerated / BatchNorm1dGenerated (modules/generated.py:7-96),
LocationSensitiveAttention (modules/attention.py), forward values and gradients through the library ops.  What the reference modules
computed on the seeded set-up of each test is stored in tests/golden/modules_*.npz (tests/golden/make_golden_modules.py); the tests
regenerate the same weights and inputs (checked against the stored digests) and compare the library's results with it."""
import pytest
import torch

from helpers import assert_close, ModuleGolden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module', autouse=True)
def _built():
    import __graft_entry__ as entry
    entry.build()
    assert torch.cuda.is_available()


def _copy_params(dst, src):
    dst.load_state_dict(src.state_dict(), strict=True)


@pytest.mark.parametrize('kind', ['zoneout', 'dropout'])
def test_lstm_cells_match_reference_eval_mode(kind):
    from multilingual_text_to_speech_b200.modules.layers import ZoneoutLSTMCell, DropoutLSTMCell
    gold = ModuleGolden('modules_lstm', kind)
    torch.manual_seed(3)
    I, H, B = 544, 1024, 7
    make = (lambda: ZoneoutLSTMCell(I, H, 0.1, 0.1)) if kind == 'zoneout' else (lambda: DropoutLSTMCell(I, H, 0.1))
    ref = make().eval()                # the reference cell's weights: same class layout, same seed, same draw order
    own = make().eval()
    _copy_params(own, ref)
    for n, p in ref.named_parameters():
        gold.check_digest(n, p)
    own = own.cuda()
    x, h, c = torch.randn(B, I), torch.randn(B, H), torch.randn(B, H)
    xo, ho, co = (t.cuda().requires_grad_(True) for t in (x, h, c))
    h2, c2 = own(xo, ho, co)
    gold.assert_close(h2, 'h', 1e-3, 1e-5); gold.assert_close(c2, 'c', 1e-3, 1e-5)
    gh, gc = torch.randn(B, H), torch.randn(B, H)
    for n, t in (('x', x), ('h', h), ('c', c), ('gh', gh), ('gc', gc)):
        gold.check_digest(n, t)
    ((h2 * gh.cuda()).sum() + (c2 * gc.cuda()).sum()).backward()
    for name, a in (('dx', xo), ('dh', ho), ('dc', co)):
        gold.assert_close(a.grad, name, 2e-3, 1e-5)
    for n, p in own.named_parameters():
        gold.assert_close(p.grad, 'd' + n, 2e-3, 1e-4 * float(gold['absmax.d' + n]))


def test_zoneout_cell_train_mode_with_masks():
    """Training mode: h = (1 - z) * dropout(h' - h, z) + h with explicit keep masks (reference layers.py:29-30 with F.dropout's mask)."""
    from multilingual_text_to_speech_b200.modules.layers import ZoneoutLSTMCell
    from multilingual_text_to_speech_b200.rng import MaskSource
    torch.manual_seed(4)
    I, H, B, z = 96, 128, 5, 0.1
    cell = ZoneoutLSTMCell(I, H, z, z).train()
    x, h, c = torch.randn(B, I), torch.randn(B, H), torch.randn(B, H)
    mh, mc = (torch.rand(B, H) >= z).float(), (torch.rand(B, H) >= z).float()
    xr, hr, cr = (t.clone().double().requires_grad_(True) for t in (x, h, c))
    w = {k: v.detach().double() for k, v in cell.state_dict().items()}
    g = xr @ w['weight_ih'].t() + w['bias_ih'] + hr @ w['weight_hh'].t() + w['bias_hh']
    i_, f_, g_, o_ = g.chunk(4, 1)
    cn = torch.sigmoid(f_) * cr + torch.sigmoid(i_) * torch.tanh(g_)
    hn = torch.sigmoid(o_) * torch.tanh(cn)
    h1 = (1 - z) * (mh.double() * (hn - hr) / (1 - z)) + hr
    c1 = (1 - z) * (mc.double() * (cn - cr) / (1 - z)) + cr
    cell = cell.cuda()
    xo, ho, co = (t.cuda().requires_grad_(True) for t in (x, h, c))
    MaskSource.use_tape({'cell_h': mh, 'cell_c': mc})
    try:
        h2, c2 = cell(xo, ho, co)
    finally:
        MaskSource.use_tape(None)
    assert_close(h2, h1, 1e-3, 1e-5, 'h'); assert_close(c2, c1, 1e-3, 1e-5, 'c')
    gh, gc = torch.randn(B, H), torch.randn(B, H)
    ((h1 * gh.double()).sum() + (c1 * gc.double()).sum()).backward()
    ((h2 * gh.cuda()).sum() + (c2 * gc.cuda()).sum()).backward()
    for name, a, b in (('dx', xo, xr), ('dh', ho, hr), ('dc', co, cr)):
        assert_close(a.grad, b.grad, 2e-3, 1e-5, name)


@pytest.mark.parametrize('train', [True, False])
def test_generated_conv_and_batchnorm_match_reference(train):
    from multilingual_text_to_speech_b200.modules.generated import Conv1dGenerated, BatchNorm1dGenerated
    gold = ModuleGolden('modules_generated', 'train' if train else 'eval')
    torch.manual_seed(5)
    G, gd, bn, Cin, Cout, k, dil, NB, L = 3, 6, 4, 8, 12, 3, 2, 4, 21
    e = torch.randn(G, gd)
    x = torch.randn(NB, G * Cin, L + (k - 1) * dil)          # the caller pads (ConvBlockGenerated pads before the convolution)
    # the reference modules' weights: same class layout, same seed, same draw order
    rc = Conv1dGenerated(gd, bn, G * Cin, G * Cout, k, padding=0, dilation=dil, groups=G, bias=False)
    oc = Conv1dGenerated(gd, bn, G * Cin, G * Cout, k, padding=0, dilation=dil, groups=G, bias=False).train(train)
    _copy_params(oc, rc)
    rb = BatchNorm1dGenerated(gd, bn, G * Cout, groups=G)
    ob = BatchNorm1dGenerated(gd, bn, G * Cout, groups=G).train(train)
    _copy_params(ob, rb)
    for n, p in [('conv.' + n, p) for n, p in rc.named_parameters()] + [('bn.' + n, p) for n, p in rb.named_parameters()]:
        gold.check_digest(n, p)
    oc, ob = oc.cuda(), ob.cuda()
    eo, xo = e.cuda().requires_grad_(True), x.cuda().requires_grad_(True)
    y2 = oc(eo, xo)                                          # un-padded ("valid") convolution, as in the reference
    assert y2.shape == gold['y'].shape and y2.shape[2] == L
    gold.assert_close(y2, 'y', 1e-3, 1e-5)
    z2 = ob(eo, y2)
    gold.assert_close(z2, 'z', 1e-3, 1e-4)
    gz = torch.randn_like(z2, device='cpu')
    for n, t in (('e', e), ('x', x), ('gz', gz)):
        gold.check_digest(n, t)
    (z2 * gz.cuda()).sum().backward()
    gold.assert_close(eo.grad, 'de', 3e-3, 1e-4 * float(gold['absmax.de']))
    gold.assert_close(xo.grad, 'dx', 3e-3, 1e-4 * float(gold['absmax.dx']))
    for n, p in [('conv.' + n, p) for n, p in oc.named_parameters()] + [('bn.' + n, p) for n, p in ob.named_parameters()]:
        gold.assert_close(p.grad, 'd' + n, 3e-3, 2e-4 * float(gold['absmax.d' + n]) + 1e-9)
    if train:
        gold.assert_close(ob.running_mean, 'running_mean', 1e-3, 1e-6)
        gold.assert_close(ob.running_var, 'running_var', 1e-3, 1e-6)
        assert int(ob.num_batches_tracked) == int(gold['num_batches_tracked']) == 1


def test_attention_module_forward_and_autograd_match_reference():
    """LocationSensitiveAttention.reset + three forward steps (attention.py:23-28, 39-45, 67-86) with gradients through the carried
    cumulative weights, against the reference module."""
    from multilingual_text_to_speech_b200.modules.attention import LocationSensitiveAttention
    gold = ModuleGolden('modules_attention', 'attention')
    torch.manual_seed(7)
    B, L, M, D, A, C, K = 5, 37, 288, 1024, 128, 32, 31
    ref = LocationSensitiveAttention(K, C, False, A, D, M)   # the reference module's weights: same layout, seed and draw order
    own = LocationSensitiveAttention(K, C, False, A, D, M)
    with torch.no_grad():
        for prm in ref.parameters():
            prm.mul_(3.0)
    _copy_params(own, ref)
    for n, p in ref.named_parameters():
        gold.check_digest(n, p)
    own = own.cuda()
    lens = torch.tensor([37, 30, 37, 12, 25])
    mask = torch.arange(L)[None, :] < lens[:, None]
    memory = torch.randn(B, L, M)
    queries = [torch.randn(B, D) for _ in range(3)]
    gold.check_digest('memory', memory)
    for step in range(3):
        gold.check_digest(f'query{step}', queries[step])
    mo = memory.cuda().requires_grad_(True); qo = [q.cuda().requires_grad_(True) for q in queries]
    own.reset(mo, B, L, mo.device)
    gen = torch.Generator().manual_seed(1)
    loss_o = 0.0
    for step in range(3):
        c2, w2 = own(qo[step], mo, mask.cuda(), None)
        gold.assert_close(w2, f'weights{step}', 1e-3, 1e-6)
        gold.assert_close(c2, f'context{step}', 1e-3, 1e-5)
        gc, gw = torch.randn(B, M, generator=gen), torch.randn(B, L, generator=gen)
        loss_o = loss_o + (c2 * gc.cuda()).sum() + (w2 * gw.cuda()).sum()
    loss_o.backward()
    gold.assert_close(mo.grad, 'dmemory', 3e-3, 1e-4 * float(gold['absmax.dmemory']))
    for step in range(3):
        gold.assert_close(qo[step].grad, f'dquery{step}', 3e-3, 1e-4 * float(gold[f'absmax.dquery{step}']))
    for n, p in own.named_parameters():
        gold.assert_close(p.grad, 'd' + n, 3e-3, 2e-4 * float(gold['absmax.d' + n]))
