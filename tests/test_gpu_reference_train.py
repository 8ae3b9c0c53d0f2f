""""train.py calls into it unchanged" (north_star, SURVEY 8b): the reference's OWN `train()` function body
(oracle/_ref/train.py:29-95, a byte-identical copy of the original project's train.py installed by build()) drives THIS package for two optimisation steps.

train.py is imported as it is; only what it imports at module level is substituted:
  params.params, modules.tacotron2, utils (lengths_to_mask, to_gpu)  -> this package (the two import lines INTEGRATION.md names)
  dataset.dataset, utils.audio, utils.text, utils.logging, utils.samplers -> inert stubs (corpus readers, DSP, TensorBoard: none is on the
  hot path and their third-party dependencies are absent from the image)
Checks: the loop runs (forward, TacotronLoss, classifier accuracy, backward, clip_grad_norm_, Adam step, criterion.update_states), the
parameters move, the losses it logs are finite, and a second identical batch gives a different (lower or higher, but changed) loss.
"""
import importlib.util
import os
import sys
import types
import pytest
import torch

from helpers import ROOT

pytestmark = pytest.mark.gpu
TRAIN_PY = os.path.join(ROOT, 'oracle', '_ref', 'train.py')


@pytest.fixture(scope='module', autouse=True)
def _built():
    import __graft_entry__ as entry
    entry.build()
    assert torch.cuda.is_available()


def _import_reference_train(logged):
    from multilingual_text_to_speech_b200.params import params as own_params
    from multilingual_text_to_speech_b200.modules import tacotron2 as own_tacotron2
    from multilingual_text_to_speech_b200 import utils as own_utils
    import multilingual_text_to_speech_b200.modules as own_modules

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    class Logger:
        @staticmethod
        def training(train_step, losses, gradient, learning_rate, duration, classifier):
            logged.append((train_step, {k: float(v) for k, v in losses.items()}, float(gradient), learning_rate, classifier))

    utils_pkg = stub('utils', lengths_to_mask=own_utils.lengths_to_mask, to_gpu=own_utils.to_gpu, __path__=[])
    utils_pkg.audio, utils_pkg.text = stub('utils.audio'), stub('utils.text')
    subst = {
        'params': stub('params', __path__=[]), 'params.params': own_params,
        'modules': own_modules, 'modules.tacotron2': own_tacotron2,
        'utils': utils_pkg, 'utils.audio': utils_pkg.audio, 'utils.text': utils_pkg.text,
        'utils.logging': stub('utils.logging', Logger=Logger),
        'utils.samplers': stub('utils.samplers', RandomImbalancedSampler=object, PerfectBatchSampler=object),
        'dataset': stub('dataset', __path__=[]),
        'dataset.dataset': stub('dataset.dataset', TextToSpeechDatasetCollection=object, TextToSpeechCollate=object),
    }
    saved = {k: sys.modules.get(k) for k in subst}
    sys.modules.update(subst)
    try:
        spec = importlib.util.spec_from_file_location('reference_train_py', TRAIN_PY)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


@pytest.mark.skipif(not os.path.exists(TRAIN_PY), reason='oracle/_ref (the unmodified reference) is not installed')
@pytest.mark.parametrize('config', ['generated_switching', 'ljspeech'])
def test_reference_train_function_runs_on_this_package(config):
    from multilingual_text_to_speech_b200 import configs
    from multilingual_text_to_speech_b200.modules.tacotron2 import Tacotron, TacotronLoss
    from multilingual_text_to_speech_b200.rng import MaskSource
    logged = []
    train_py = _import_reference_train(logged)
    small = dict(embedding_dimension=32, encoder_dimension=32, prenet_dimension=24, attention_dimension=16, attention_kernel_size=7,
                 attention_location_dimension=8, decoder_dimension=48, postnet_dimension=32, num_mels=12, reversal_classifier_dim=16,
                 speaker_embedding_dimension=8)
    hp = configs.apply(config, speakers=3, **small)
    assert train_py.hp is hp                                   # train.py reads THIS package's Params
    G = max(hp.language_number, 1)
    B, L, T = 2 * G, 14, 20
    torch.manual_seed(0)
    MaskSource.manual_seed(1)
    model = Tacotron().cuda()
    optimizer = torch.optim.Adam(model.parameters(), lr=hp.learning_rate, weight_decay=hp.weight_decay)
    criterion = TacotronLoss(hp.guided_attention_steps, hp.guided_attention_toleration, hp.guided_attention_gain)
    g = torch.Generator().manual_seed(3)
    lens = torch.sort(torch.randint(L // 2, L + 1, (B,), generator=g), descending=True).values; lens[0] = L
    text = torch.randint(1, hp.symbols_count() + 3, (B, L), generator=g)
    for b in range(B):
        text[b, lens[b]:] = 0
    tlens = torch.full((B,), T)
    stop = torch.zeros(B, T); stop[:, -hp.stop_frames:] = 1
    batch = (text, lens, torch.randn(B, hp.num_mels, T, generator=g), None, tlens, stop,
             torch.randint(0, 3, (B,), generator=g) if hp.multi_speaker else None, (torch.arange(B) % G) if hp.multi_language else None)
    before = [p.detach().clone() for p in model.parameters()]
    g_before = criterion._g
    train_py.train(0, 0, [batch, batch], model, criterion, optimizer)       # logging_start_epoch 0 -> Logger.training is called
    assert len(logged) == 2
    for step, losses, grad, lr, cla in logged:
        assert all(v == v and abs(v) < 1e4 for v in losses.values()) and grad == grad and grad > 0
        assert {'mel_pre', 'mel_pos', 'stop_token', 'guided_att'} <= set(losses)
        if hp.reversal_classifier:
            assert 'lang_class' in losses and 0.0 <= cla <= 1.0
    assert logged[0][1]['mel_pre'] != logged[1][1]['mel_pre']                   # the optimiser step changed the model
    moved = sum(int(not torch.equal(p, q)) for p, q in zip(model.parameters(), before))
    assert moved == len(before), f'only {moved} of {len(before)} parameter tensors were updated'
    assert criterion._g == g_before * hp.guided_attention_gain ** 2          # update_states ran once per step
