"""CPU tests of the host-side mirror: registry, config system, checkpoint layout."""
import os

import numpy as np
import pytest
import torch

from neuralsvb_b200.utils import audio, hparams as HP, synthetic as S
from neuralsvb_b200.vocoders.base_vocoder import VOCODERS, BaseVocoder, get_vocoder_cls, register_vocoder


def test_registry_names_and_dotted_path():
    import neuralsvb_b200.vocoders  # noqa: F401
    from neuralsvb_b200.vocoders.hifigan import HifiGAN
    assert VOCODERS['HifiGAN'] is HifiGAN and VOCODERS['hifigan'] is HifiGAN
    assert get_vocoder_cls({'vocoder': 'hifigan'}) is HifiGAN
    assert get_vocoder_cls({'vocoder': 'neuralsvb_b200.vocoders.hifigan.HifiGAN'}) is HifiGAN

    @register_vocoder
    class Dummy(BaseVocoder):
        pass
    assert get_vocoder_cls({'vocoder': 'dummy'}) is Dummy
    with pytest.raises(NotImplementedError):
        Dummy().spec2wav(None)


def test_hparams_chain_override_and_cli(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    (tmp_path / 'a').mkdir()
    (tmp_path / 'base.yaml').write_text('x: 1\nnest: {p: 1, q: 2}\nlst: [1, 2]\nflag: false\nname: abc\n')
    (tmp_path / 'a' / 'mid.yaml').write_text('base_config: ../base.yaml\nx: 2\nnest: {q: 3}\n')
    (tmp_path / 'a' / 'top.yaml').write_text('base_config:\n  - ./mid.yaml\ny: 5.5\n')
    hp = HP.set_hparams('a/top.yaml', hparams_str='lst=[3 4 5],flag=True,nest.p=7,y=1.5,name=zz',
                        print_hparams=False, global_hparams=False)
    assert hp['x'] == 2 and hp['nest'] == {'p': 7, 'q': 3} and hp['lst'] == [3, 4, 5]
    assert hp['flag'] is True and hp['y'] == 1.5 and hp['name'] == 'zz' and hp['work_dir'] == ''
    # exp_name -> config.yaml snapshot written and merged back on the next run
    HP.set_hparams('a/top.yaml', exp_name='e1', hparams_str='x=9', print_hparams=False, global_hparams=True)
    assert os.path.exists('checkpoints/e1/config.yaml') and HP.hparams['x'] == 9
    hp2 = HP.set_hparams('a/top.yaml', exp_name='e1', print_hparams=False, global_hparams=False)
    assert hp2['x'] == 9 and hp2['work_dir'] == 'checkpoints/e1'


def test_hparams_resolves_reference_yaml_like_the_reference(golden_dir, tmp_path, monkeypatch):
    """base_config chains of the reference's egs/ tree resolve to the dict the reference's set_hparams returned
    (tests/golden/hparams.json, written by oracle/gen_golden.py gen_hparams: the YAML files parsed, and the resolved dicts)."""
    import json
    import yaml
    gold = json.load(open(os.path.join(golden_dir, 'hparams.json')))
    for rel, content in gold['files'].items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(yaml.safe_dump(content, sort_keys=False))
    monkeypatch.chdir(tmp_path)
    assert len(gold['cases']) == 2
    for case in gold['cases']:
        a = HP.set_hparams(case['config'], hparams_str=case['hparams_str'], print_hparams=False, global_hparams=False)
        assert a == case['resolved']


def test_generator_state_dict_layout_is_the_checkpoint_contract():
    from neuralsvb_b200.modules.hifigan.hifigan import HifiGanGenerator
    h = S.hifigan_config()
    m = HifiGanGenerator(h)
    keys = list(m.state_dict())
    assert 'conv_pre.weight_g' in keys and 'ups.0.weight_v' in keys and 'm_source.l_linear.weight' in keys
    assert 'resblocks.11.convs2.2.weight_v' in keys and 'noise_convs.3.bias' in keys and len(keys) == 244
    assert tuple(m.state_dict()['ups.0.weight_g'].shape) == (512, 1, 1)     # weight norm over dim 0 = Cin
    sd = S.make_generator_state_dict(h)
    m.load_state_dict(sd, strict=True)
    assert sum(v.numel() for v in sd.values()) == 13_954_154 or sum(v.numel() for v in sd.values()) > 13_900_000


def test_mel_basis_and_pad_helpers():
    fb = audio.mel_filterbank(22050, 1024, 80, 80, 7600)
    assert fb.shape == (80, 513) and fb.dtype == np.float32 and (fb.sum(1) > 0).all()
    x = np.zeros(44100, np.float32)
    assert audio.librosa_pad_lr(x, 1024, 256, 1) == (0, 173 * 256 - 44100)
    l, r = audio.librosa_pad_lr(x, 1024, 256, 2)
    assert l + r == 173 * 256 - 44100


def test_vocoder_training_task_wiring_on_cpu(monkeypatch, tmp_path):
    """egs/vocoder_train_synthetic.yaml -> HifiGanTask: modules with the reference's parameter names, two AdamW optimizers
    over disjoint parameter sets (the trainer's two-optimizer contract), synthetic batches of the yaml's shape.
    No kernel runs here (no GPU): this pins the host-side wiring only."""
    from neuralsvb_b200.tasks.vocoder.hifigan import HifiGanTask
    monkeypatch.chdir(tmp_path)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hp = HP.set_hparams(config=os.path.join(root, 'egs/vocoder_train_synthetic.yaml'), exp_name='',
                        hparams_str='max_sentences=3,max_samples=4096,num_train_batches=2', print_hparams=False)
    assert hp['task_cls'].endswith('HifiGanTask') and hp['lambda_mel'] == 5.0 and hp['upsample_rates'] == [8, 8, 2, 2]
    HP.hparams['infer'] = False
    task = HifiGanTask()
    assert task.build_model() is None
    gen_names = set(dict(task.model_gen.named_parameters()))
    assert gen_names == set(S.make_generator_state_dict(S.hifigan_config(), 1))         # the reference's checkpoint keys
    assert set(task.model_disc['mpd'].state_dict()) == set(S.make_mpd_state_dict(1))
    assert set(task.model_disc['msd'].state_dict()) == set(S.make_msd_state_dict(1))
    og, od = task.configure_optimizers()
    ids_g = {id(p) for g in og.param_groups for p in g['params']}
    ids_d = {id(p) for g in od.param_groups for p in g['params']}
    assert ids_g and ids_d and not (ids_g & ids_d)
    assert og.defaults['betas'] == (0.8, 0.99) and abs(og.defaults['lr'] - 2e-4) < 1e-12
    batches = task.train_dataloader()
    assert len(batches) == 2 and tuple(batches[0]['wavs'].shape) == (3, 1, 4096) and tuple(batches[0]['f0'].shape) == (3, 16)


def test_tensor_core_eligibility_of_discriminator_layers():
    from neuralsvb_b200.modules.hifigan import discriminators as D
    # MPD: (cin, cout) with k 5, stride 3 (1 for the last), pad 2
    assert not D.tc_eligible(1, 32, 5, 3, 1, 2, 1)             # 1 input channel: fp32 kernel
    assert D.tc_eligible(32, 128, 5, 3, 1, 2, 1) and D.tc_eligible(512, 1024, 5, 3, 1, 2, 1)
    assert D.tc_eligible(1024, 1024, 5, 1, 1, 2, 1)            # stride 1, 'same' padding
    assert not D.tc_eligible(1024, 1, 3, 1, 1, 1, 1)           # conv_post: one output channel
    # MSD: every grouped k = 41 layer (hifigan.py:263-267) tiles the tensor-core kernel in polyphase form; 1 -> 128 k15 does not
    from neuralsvb_b200.utils.synthetic import MSD_LAYERS
    for cin, cout, k, s, g, p in MSD_LAYERS[1:6]:
        assert D.tc_eligible(cin, cout, k, s, 1, p, g), (cin, cout, k, s, g)
    assert not D.tc_eligible(1, 128, 15, 1, 1, 7, 1) and D.tc_eligible(1024, 1024, 5, 1, 1, 2, 1)
    assert not D.tc_eligible(128, 128, 40, 2, 1, 20, 4)        # ceil(40 / 2) = 20 taps: even, no centred form
    D.USE_TC_GROUPED = False
    try:
        assert not D.tc_eligible(128, 128, 41, 2, 1, 20, 4)
    finally:
        D.USE_TC_GROUPED = True
    assert not D.tc_eligible(1024, 1024, 5, 1, 1, 1, 1)        # not 'same' padding


def test_indexed_dataset_format_and_vocoder_loader(tmp_path):
    """N3: the reference's on-disk format ({path}.data = concatenated pickles, {path}.idx = np.save'd offsets,
    utils/indexed_datasets.py:7-54) and the batch loader on top of it: frame-aligned crops, [B,1,n] / [B,T,80] / [B,T]
    tensors, the global batch sharded batch[rank::world] with disjoint shards, uneven tails dropped."""
    import pickle
    import numpy as np
    from neuralsvb_b200.tasks.vocoder.dataset_utils import VocoderBatchLoader
    from neuralsvb_b200.utils.indexed_datasets import IndexedDataset, IndexedDatasetBuilder
    hop, n_items = 16, 11
    rs = np.random.RandomState(0)
    path = str(tmp_path / 'train')
    b = IndexedDatasetBuilder(path)
    items = []
    for i in range(n_items):
        T = 20 + 3 * i
        mel = rs.randn(T, 80).astype(np.float32)
        wav = (np.arange(T * hop) % hop + 100 * i).astype(np.float16)          # sample value encodes (item, position in frame)
        f0 = np.arange(T, dtype=np.float32) + 1000 * i
        items.append({'item_name': f'it{i}', 'mel': mel, 'wav': wav, 'f0': f0, 'len': T, 'sec': T * hop / 22050})
        b.add_item(items[-1])
    b.finalize()
    # byte layout of the reference: offsets index concatenated pickles
    off = np.load(path + '.idx', allow_pickle=True).item()['offsets']
    raw = open(path + '.data', 'rb').read()
    assert len(off) == n_items + 1 and off[-1] == len(raw)
    assert pickle.loads(raw[off[3]:off[4]])['item_name'] == 'it3'
    ds = IndexedDataset(path)
    assert len(ds) == n_items and np.array_equal(ds[5]['mel'], items[5]['mel'])
    with pytest.raises(IndexError):
        ds[n_items]
    seen = []
    for rank in range(2):
        ld = VocoderBatchLoader(path, hop, max_samples=8 * hop, max_sentences=2, rank=rank, world=2, seed=3, pin=False)
        assert len(ld) == n_items // 4
        batches = list(ld)
        assert len(batches) == 2                                               # 11 items, global batch 4: the tail of 3 is dropped
        for bt in batches:
            assert bt['wavs'].shape == (2, 1, 8 * hop) and bt['mels'].shape == (2, 8, 80) and bt['f0'].shape == (2, 8)
            for j, name in enumerate(bt['item_names']):
                i = int(name[2:])
                s = int(bt['f0'][j, 0]) - 1000 * i                             # crop start frame, recovered from f0
                assert np.array_equal(bt['mels'][j].numpy(), items[i]['mel'][s:s + 8])
                assert np.array_equal(bt['wavs'][j, 0].numpy(), items[i]['wav'][s * hop:(s + 8) * hop].astype(np.float32))
            seen.append((rank, tuple(bt['item_names'])))
    r0 = {n for r, names in seen if r == 0 for n in names}
    r1 = {n for r, names in seen if r == 1 for n in names}
    assert not (r0 & r1) and len(r0) == len(r1) == 4                           # disjoint shards of the same global batches


# ---- SVB acoustic model drop-ins (SURVEY 8(f) N1): host-side contracts that need no GPU
def test_acoustic_modules_refuse_cpu_tensors_and_training_mode():
    """No CPU / PyTorch fallback in the product (DESIGN section 1): the drop-in classes raise instead of silently computing elsewhere."""
    import pytest
    import torch
    from neuralsvb_b200.modules.fastspeech.fs2_vae import WN, FVAEDecoder
    from neuralsvb_b200.modules.voice_conversion.vc_modules import VCASR
    wn = WN(64, 3, 1, 2).eval()
    with pytest.raises(RuntimeError, match='no CPU path'):
        with torch.no_grad():
            wn(torch.zeros(1, 64, 16))
    dec = FVAEDecoder(16, 64, 80, 3, 2).eval()
    with pytest.raises(RuntimeError, match='no CPU path'):
        with torch.no_grad():
            dec(torch.zeros(1, 16, 4), 1, None)
    asr = VCASR(80, 80, hidden_size=64, asr_enc_layers=1, mel_strides=[2, 1, 1], asr_last_norm=False)
    with pytest.raises(RuntimeError, match='inference only'):
        asr.train()(torch.zeros(1, 8, 80))
    with pytest.raises(RuntimeError, match='no CPU path'):
        with torch.no_grad():
            asr.eval()(torch.zeros(1, 8, 80))
    with pytest.raises(NotImplementedError):
        WN(64, 3, 1, 2, share_cond_layers=True)


def test_vc_asr_ignores_the_token_decoder_of_a_reference_checkpoint():
    """vc_modules.py:69-74 of the reference also owns an ASR token decoder (training head); its checkpoint keys must not break loading."""
    import torch
    from neuralsvb_b200.modules.voice_conversion.vc_modules import VCASR
    from neuralsvb_b200.utils import synthetic as S
    sd = S.make_vc_asr_state_dict(1234)
    sd['asr_decoder.layers.0.self_attn.in_proj_weight'] = torch.zeros(3)
    sd['token_embed.weight'] = torch.zeros(80, 256)
    m = VCASR(80, 80, hidden_size=256, asr_enc_layers=2, mel_strides=[2, 1, 1], asr_last_norm=False)
    m.load_state_dict(sd, strict=True)
    assert torch.equal(m.content_encoder.encoder_layers[1].self_attn.pos_bias_u, sd['content_encoder.encoder_layers.1.self_attn.pos_bias_u'])
    assert isinstance(m.content_encoder.layer_norm, torch.nn.Linear)          # asr_last_norm false (vc_ppg.yaml:16)
    assert isinstance(VCASR(80, 80, hidden_size=64, asr_enc_layers=1, mel_strides=[2, 1, 1], asr_last_norm=True).content_encoder.layer_norm,
                      torch.nn.LayerNorm)


def test_wn_state_dict_names_before_and_after_weight_norm_removal():
    from neuralsvb_b200.modules.fastspeech.fs2_vae import WN
    from neuralsvb_b200.utils import synthetic as S
    m = WN(64, 3, 2, 3, gin_channels=32)
    sd = S.make_wn_state_dict(64, 3, 3, 32, 1234)
    assert set(m.state_dict()) == set(sd)
    m.load_state_dict(sd, strict=True)
    m.remove_weight_norm()
    names = set(m.state_dict())
    assert 'cond_layer.weight' in names and 'in_layers.2.weight' in names and not any(k.endswith(('weight_g', 'weight_v')) for k in names)
    assert tuple(m.state_dict()['res_skip_layers.2.weight'].shape) == (64, 64, 1)      # the last layer has no skip half (fs2_vae.py:52-55)
