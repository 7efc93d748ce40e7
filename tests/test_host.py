"""CPU: host-side logic -- gin subset reader, InferenceModel config surface, parameter tree,
C-ABI header vs exported symbols (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from music_spectrogram_diffusion_b200 import (_native, audio_codecs, config, engine, gin_lite,
                                              inference, weights)

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GIN = os.path.join(HERE, 'golden', 'base_with_context.gin')


def test_gin_lite_macros_scopes_blocks():
  g = gin_lite.parse_config(open(GIN).read())
  assert g.query_macro('TASK_FEATURE_LENGTHS') == {'inputs': 2048, 'targets': 256,
                                                   'targets_context': 256}
  assert g.query_macro('%NUM_VELOCITY_BINS') == 1
  model = g.macros['MODEL']
  assert isinstance(model, gin_lite.ConfigurableRef) and model.evaluate
  assert model.name.endswith('ContextDiffusionModel')
  t5 = g.bindings_for('network.T5Config')
  assert t5['emb_dim'] == 768 and t5['mlp_activations'] == ('gelu', 'linear')
  assert isinstance(t5['vocab_size'], gin_lite.ConfigurableRef)
  assert g.bindings_for('diffusion_utils.DiffusionSchedule', 'sampler')['num_steps'] == 1000
  assert 'num_steps' not in g.bindings_for('diffusion_utils.DiffusionSchedule', 'train')


def test_gin_lite_overrides_and_continuations():
  text = open(GIN).read() + '''
diffusion_utils.ClassifierFreeGuidanceConfig.eval_condition_weight = 2.0
network.T5Config.mlp_activations = (
    'gelu',
    'linear',
)  # trailing comment
'''
  g = gin_lite.parse_config(text)
  assert g.bindings_for('diffusion_utils.ClassifierFreeGuidanceConfig') == {
      'eval_condition_weight': 2.0}
  assert g.bindings_for('network.T5Config')['mlp_activations'] == ('gelu', 'linear')
  with pytest.raises(ValueError):
    gin_lite.parse_config('this is not gin')


def test_inference_model_config_surface(tmp_path):
  gin_config = inference.parse_training_gin_file(
      GIN, ['diffusion_utils.ClassifierFreeGuidanceConfig.eval_condition_weight = 2.0'])
  m = inference.InferenceModel('synthetic:0', gin_config, batch_size=3)
  assert m.sequence_length == {'inputs': 2048, 'targets': 256, 'targets_context': 256}
  assert (m.inputs_length, m.targets_length, m.targets_context_length) == (2048, 256, 256)
  assert m.batch_size == 3
  ac = m.audio_codec
  assert (ac.n_dims, ac.hop_size, ac.sample_rate, ac.frame_rate) == (128, 320, 16000, 50)
  assert m.input_shapes == {
      'encoder_input_tokens': (3, 2048), 'decoder_target_tokens': (3, 256, 128),
      'encoder_continuous_inputs': (3, 256, 128), 'encoder_continuous_mask': (3, 256)}
  assert m.input_types['encoder_input_tokens'] == np.int32
  t5 = m.model.module_config
  assert (t5.vocab_size, t5.emb_dim, t5.num_heads, t5.mlp_dim) == (1536, 768, 12, 2048)
  d = m.model.diffusion_config
  assert d.sampler.schedule.num_steps == 1000 and d.sampler.name == 'ddpm'
  assert d.classifier_free_guidance.eval_condition_weight == 2.0
  assert 'encoder_continuous_mask' in m.model.FEATURE_CONVERTER_CLS.MODEL_FEATURES
  assert m.partitioner.partition(len) is len   # the colab monkey-patches this attribute
  cfg = engine.make_msd_config(t5, d, 2048, 256, 256, 3)
  assert (cfg.vocab_size, cfg.num_steps, cfg.sampler, cfg.context_positions) == (1536, 1000, 0, 1)
  assert abs(cfg.feature_min - np.log(1e-5)) < 1e-6 and cfg.feature_max == 4.0


def test_vocab_size_rule():
  """vocabularies.py:118-144, 279-281: 1388 codec classes + 3 + 100 -> 1536."""
  c = inference.build_codec(num_velocity_bins=1)
  assert c.num_classes == 1388 and inference.num_embeddings(c) == 1536
  assert inference.num_embeddings(inference.build_codec(num_velocity_bins=127)) == 1664
  # the reference's Codec surface (event_codec.py:64-112) on the same object
  assert c.max_shift_steps == 1000 and c.steps_per_second == 100 and c.is_shift_event_index(1000)
  assert not c.is_shift_event_index(1001) and c.event_type_range('pitch') == (1001, 1128)
  ev = c.decode_event_index(c.encode_event(('program', 40)))
  assert (ev.type, ev.value) == ('program', 40)


def test_unsupported_configs_fail_loudly():
  t5 = config.t5_base()
  d = config.DiffusionConfig()
  t5.mlp_activations = ('relu',)
  with pytest.raises(NotImplementedError):
    engine.make_msd_config(t5, d, 2048, 256, 256, 1)
  t5 = config.t5_base()
  t5.decoder_cross_attend_style = 'sum_cross_attends'
  assert engine.make_msd_config(t5, d, 2048, 256, 256, 1).cross_attend_style == 1
  t5.decoder_cross_attend_style = 'product'
  with pytest.raises(ValueError, match='Unknown decoder_cross_attend_style'):
    engine.make_msd_config(t5, d, 2048, 256, 256, 1)


def test_param_tree_matches_reference_counts():
  """SURVEY F6 / App. C: 411.67 M (base), 104.04 M (small); decoder split."""
  shapes = weights.param_shapes(config.t5_base(), 2048, 256, 256)
  assert weights.num_params(shapes) == 411_665_664
  dec = [(n, s) for n, s in shapes if n.startswith('decoder/')]
  film = sum(int(np.prod(s)) for n, s in dec if 'FiLMLayer' in n)
  assert film == 24 * 3072 * 1536
  assert weights.num_params(weights.param_shapes(config.t5_small(), 2048, 256, 256)) == 104_035_840
  names = [n for n, _ in shapes]
  assert 'decoder/layers_3/MultiHeadDotProductAttention_0/query/kernel' in names
  assert 'continuous_encoder/input_proj/kernel' in names
  assert len(set(names)) == len(names)


def test_synthetic_params_roundtrip(tmp_path):
  t5 = config.t5_tiny()
  p = weights.synthetic_params(t5, 128, 128, 128, seed=3)
  q = weights.synthetic_params(t5, 128, 128, 128, seed=3)
  assert all(np.array_equal(p[k], q[k]) for k in p)
  path = str(tmp_path / 'w.npz')
  weights.save_npz(path, p)
  r = weights.load_npz(path)
  assert set(r) == set(p) and all(np.array_equal(p[k], r[k]) for k in p)


def test_audio_codec_scaling():
  ac = audio_codecs.MelGAN()
  f = np.array([np.log(1e-5), 0.0, 4.0, 7.0], np.float32)
  s = ac.scale_features(f, clip=True)
  np.testing.assert_allclose(s[[0, 2, 3]], [-1.0, 1.0, 1.0], atol=1e-6)
  np.testing.assert_allclose(ac.scale_to_features(s)[:3], f[:3], atol=1e-5)
  with pytest.raises(NotImplementedError):
    ac.decode(f)


def test_c_abi_exports_every_declared_symbol(native_lib):
  """Every function include/msd_b200.h declares is exported, and nothing is bound twice."""
  hdr = open(os.path.join(ROOT, 'include', 'msd_b200.h')).read()
  hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
  declared = set(re.findall(r'\b(msd_[a-z0-9_]+)\s*\(', hdr))
  assert len(declared) >= 15
  bound = {name for name, _, _ in _native.SYMBOLS}
  assert declared == bound, (declared ^ bound)
  for name in declared:
    assert hasattr(native_lib, name), name
  assert native_lib.msd_abi_version() == _native.ABI_VERSION == 4
  assert isinstance(native_lib.msd_last_error(), bytes)


def test_struct_layout_matches_header():
  """msd_config (ABI 3): 17 int32, 4 float, 4 int32, 5 float, 3 int32, no padding; msd_tensor:
  ptr, ptr, int32, int64[4]."""
  assert ctypes.sizeof(_native.MsdConfig) == 17 * 4 + 4 * 4 + 4 * 4 + 5 * 4 + 4 + 4 + 4
  assert _native.MsdConfig.rng_kind.offset == 124
  assert _native.MsdConfig.precision.offset == 128
  assert _native.MsdConfig.cross_attend_style.offset == 120
  assert _native.MsdConfig.max_decoder_noise_time.offset == 68
  assert _native.MsdConfig.model_output.offset == 84
  assert _native.MsdConfig.logvar_frac.offset == 100
  assert ctypes.sizeof(_native.MsdTensor) == 8 + 8 + 8 + 32
  assert _native.MsdTensor.shape.offset == 24


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
  monkeypatch.setattr(_native, '_lib', None)
  monkeypatch.setattr(_native, 'LIB_PATH', str(tmp_path / 'nope.so'))
  with pytest.raises(_native.MsdError, match='no CPU fallback'):
    _native.load()


def test_unreachable_sampler_settings_are_refused():
  from music_spectrogram_diffusion_b200 import engine
  t5 = config.t5_tiny()
  for mutate, exc in ((lambda d: setattr(d, 'model_output', 'x0_and_eps'), NotImplementedError),
                      (lambda d: setattr(d, 'model_output', 'w'), ValueError),
                      (lambda d: setattr(d.sampler, 'logvar_type', 'medium:1.5'), ValueError),
                      (lambda d: setattr(d.sampler, 'name', 'euler'), ValueError),
                      (lambda d: setattr(d.sampler.schedule, 'name', 'sigmoid'), ValueError),
                      (lambda d: setattr(d.train_schedule, 'name', 'linear'), ValueError)):
    diff = config.DiffusionConfig()
    mutate(diff)
    with pytest.raises(exc):
      engine.make_msd_config(t5, diff, 128, 128, 128, max_batch=1)


def test_gin_bindings_reach_the_sampler_variants():
  """gin overrides of diffusion_utils.{SamplerConfig, DiffusionConfig, DiffusionSchedule} map to
  the ABI-2 fields of msd_config."""
  gin_config = inference.parse_training_gin_file(GIN, [
      "diffusion_utils.SamplerConfig.logvar_type = 'medium:0.25'",
      "diffusion_utils.SamplerConfig.name = 'ddpm'",
      "diffusion_utils.DiffusionConfig.model_output = 'v'",
      "sampler/diffusion_utils.DiffusionSchedule.name = 'linear'",
      "sampler/diffusion_utils.DiffusionSchedule.start = 1e-4",
      "sampler/diffusion_utils.DiffusionSchedule.stop = 0.02",
      "sampler/diffusion_utils.DiffusionSchedule.num_steps = 250",
  ])
  m = inference.InferenceModel('synthetic:0', gin_config, batch_size=1)
  d = m.model.diffusion_config
  assert d.sampler.schedule.name == 'linear' and d.sampler.schedule.num_steps == 250
  cfg = engine.make_msd_config(m.model.module_config, d, 2048, 256, 256, 1)
  assert (cfg.logvar_type, cfg.model_output, cfg.sampler_schedule, cfg.train_schedule) == (2, 2, 1, 0)
  assert abs(cfg.logvar_frac - 0.25) < 1e-7 and cfg.num_steps == 250
  assert abs(cfg.sampler_beta_start - 1e-4) < 1e-9 and abs(cfg.sampler_beta_stop - 0.02) < 1e-8


GIN_INCLUDE_ROOT = os.path.join(HERE, 'golden', 'gin_include')


def test_gin_lite_includes_across_files():
  """gin_lite reads the subset of gin the reference's config files use: nested includes resolved
  against a search root, macros (resolved when queried), scoped bindings, configurable references,
  bracket and backslash continuations, and later bindings overriding included ones."""
  with open(os.path.join(GIN_INCLUDE_ROOT, 'configs', 'model.gin')) as f:
    g = gin_lite.parse_config(f.read(), [GIN_INCLUDE_ROOT])
  assert g.query_macro('TASK_FEATURE_LENGTHS') == {'inputs': 2048, 'targets': 256,
                                                   'targets_context': 256}
  assert g.query_macro('NUM_VELOCITY_BINS') == 1
  assert g.query_macro('%DECODER_LAYERS') == 8
  codec, model = g.macros['AUDIO_CODEC'], g.macros['MODEL']
  assert isinstance(codec, gin_lite.ConfigurableRef) and codec.evaluate
  assert (codec.scope, codec.name) == ('', 'audio_codecs.MelGAN')
  assert model.name == 'models.ContextDiffusionModel'
  t5 = g.bindings_for('network.T5Config')
  assert t5['emb_dim'] == 512 and g.resolve(t5['num_decoder_layers']) == 8
  assert t5['mlp_activations'] == ('gelu', 'linear')
  assert t5['dropout_rate'] == 0.0
  assert isinstance(t5['vocab_size'], gin_lite.ConfigurableRef) and t5['vocab_size'].evaluate
  assert g.bindings_for('diffusion_utils.DiffusionSchedule', 'train') == {'name': 'linear'}
  assert g.bindings_for('diffusion_utils.DiffusionSchedule', 'sampler') == {'name': 'cosine',
                                                                          'num_steps': 250}
  assert g.bindings_for('diffusion_utils.DiffusionSchedule') == {'name': 'cosine'}
  with pytest.raises(FileNotFoundError):
    gin_lite.parse_config("include 'configs/missing.gin'", [GIN_INCLUDE_ROOT])


def test_reference_model_sizes_match_config():
  """The network.T5Config sizes gin_lite reads from the reference's
  gin/models/diffusion/context/*.gin (stored by tests/golden/make_reference_gin_sizes.py) are the
  ones config.py builds."""
  import json
  with open(os.path.join(HERE, 'golden', 'reference_gin_model_sizes.json')) as f:
    sizes = {name: (s['emb_dim'], s['num_heads'], s['num_decoder_layers'], s['mlp_dim'])
             for name, s in json.load(f).items()}
  assert set(sizes) == {'local_tiny', 't5_small', 't5_base', 't5_large'}
  base, small = config.t5_base(), config.t5_small()
  assert sizes['t5_base'] == (base.emb_dim, base.num_heads, base.num_decoder_layers, base.mlp_dim)
  assert sizes['t5_small'] == (small.emb_dim, small.num_heads, small.num_decoder_layers, small.mlp_dim)
  assert sizes['t5_large'] == (1024, 16, 24, 2816)


def test_header_is_plain_c(tmp_path):
  """include/msd_b200.h is the C ABI: it must compile as C99 and as C++ without any other header
  of this repository, and a C caller must see the struct layout the ctypes binding uses."""
  import shutil
  import subprocess
  if not shutil.which('gcc'):
    pytest.skip('no gcc')
  hdr = os.path.join(ROOT, 'include', 'msd_b200.h')
  for cmd in (['gcc', '-std=c99', '-Wall', '-Wextra', '-pedantic', '-fsyntax-only', '-x', 'c', hdr],
              ['g++', '-std=c++17', '-fsyntax-only', '-x', 'c++', hdr]):
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0 and not r.stderr.strip(), r.stderr
  src = tmp_path / 'layout.c'
  src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "msd_b200.h"\n'
                 'int main(void) { printf("%zu %zu %zu %zu %d\\n", sizeof(msd_config), '
                 'offsetof(msd_config, precision), sizeof(msd_tensor), offsetof(msd_tensor, shape), '
                 'MSD_B200_ABI_VERSION); return 0; }\n')
  exe = tmp_path / 'layout'
  subprocess.run(['gcc', '-std=c99', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)],
                 check=True)
  out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
  assert [int(x) for x in out] == [ctypes.sizeof(_native.MsdConfig), _native.MsdConfig.precision.offset,
                                   ctypes.sizeof(_native.MsdTensor), _native.MsdTensor.shape.offset,
                                   _native.ABI_VERSION]


def test_stale_library_is_refused(monkeypatch, native_lib):
  """load() checks msd_abi_version() against the binding (a stale .so from an older header must not
  be driven through mismatched struct layouts)."""
  monkeypatch.setattr(_native, '_lib', None)
  monkeypatch.setattr(_native, 'ABI_VERSION', _native.ABI_VERSION + 1)
  with pytest.raises(_native.MsdError, match='stale'):
    _native.load()


def test_precision_names():
  t5, d = config.t5_base(), config.DiffusionConfig()
  assert engine.make_msd_config(t5, d, 2048, 256, 256, 1).precision == 0
  assert engine.make_msd_config(t5, d, 2048, 256, 256, 1, precision='fp32_accurate').precision == 1
  with pytest.raises(ValueError, match='unknown precision'):
    engine.make_msd_config(t5, d, 2048, 256, 256, 1, precision='fp16')
