"""-m gpu: network / sampler parity of the CUDA path (through the C ABI) against the oracle."""
import numpy as np
import pytest
import torch

from music_spectrogram_diffusion_b200 import config, weights
from oracle import msd_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

T = N = C = 128


@pytest.fixture(scope='module')
def tiny():
  t5 = config.t5_tiny()
  params = weights.synthetic_params(t5, T, N, C, seed=0)
  return t5, params


def _rel(a, b):
  return ((a - b).abs().max() / b.abs().max().clamp_min(1e-6)).item()


def test_step_table(cuda_device, tiny):
  t5, params = tiny
  eng = H.build_engine(t5, T, N, C, 1, 1000, 2.0, params)
  tab = eng.step_table()
  for i in (999, 998, 500, 1):
    ref = O.sampler_coefficients(i, 1000, dtype=np.float32)
    got = tab[i]
    np.testing.assert_allclose(got[0], ref['x0_scale'], rtol=2e-3)   # fp32 tan near pi/2
    np.testing.assert_allclose(got[1], ref['eps_scale'], rtol=1e-4)
    np.testing.assert_allclose(got[2], ref['c_z'], rtol=2e-3)
    np.testing.assert_allclose(got[3], ref['c_x0'], rtol=2e-3)
    np.testing.assert_allclose(got[4], ref['sigma'], rtol=1e-4)
  assert tab[0][5] == 1.0 and tab[1][5] == 0.0
  eng.close()


def test_encode(cuda_device, tiny):
  t5, params = tiny
  B = 3
  toks, ctx, cmask = H.make_batch(B, T, C, ctx_masks=[1, 0, 1])
  cmask[2, 40:] = 0   # partially filled context -> terminal-relative roll by 40
  eng = H.build_engine(t5, T, N, C, B, 4, 2.0, params)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
             b['encoder_continuous_mask'])
  got = eng.encodings().cpu()
  oc = H.oracle_config(t5, 4, 2.0)
  cb = H.torch_batch(toks, ctx, cmask)
  encs = O.encode(O.params_to(params), oc, cb['encoder_input_tokens'],
                  O.scale_features(cb['encoder_continuous_inputs'], oc, clip=True),
                  cb['encoder_continuous_mask'])
  want = torch.cat([encs[0][0], encs[1][0]], dim=1)
  valid = torch.cat([encs[0][1], encs[1][1]], dim=1) > 0   # only unmasked positions are defined
  err = ((got - want).abs() * valid.unsqueeze(-1)).max().item()
  assert torch.isfinite(got).all()
  assert err < 6e-2, f'max err on valid positions {err}'
  eng.close()


@pytest.mark.parametrize('conditioned', [True, False])
def test_decode_eps(cuda_device, tiny, conditioned):
  t5, params = tiny
  B, steps = 2, 16
  toks, ctx, cmask = H.make_batch(B, T, C)
  eng = H.build_engine(t5, T, N, C, B, steps, 2.0, params)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
             b['encoder_continuous_mask'])
  z = torch.randn(B, N, 128, generator=torch.Generator().manual_seed(3))
  oc = H.oracle_config(t5, steps, 2.0)
  P = O.params_to(params)
  cb = H.torch_batch(toks, ctx, cmask)
  encs = O.encode(P, oc, cb['encoder_input_tokens'],
                  O.scale_features(cb['encoder_continuous_inputs'], oc, clip=True),
                  cb['encoder_continuous_mask'])
  flag = 1.0 if conditioned else 0.0
  for step_i in (steps - 1, 5, 0):
    got = eng.decode_eps(z.to(cuda_device), step_i, conditioned).cpu()
    t = np.float32(step_i + 1.0) / np.float32(steps)
    want = O.decode(P, oc, [(e * flag, m * flag) for e, m in encs], z,
                    torch.full((B,), float(t)))
    rel = ((got - want).abs().max() / want.abs().max()).item()
    assert rel < 3e-2, f'step {step_i}: rel max err {rel}'
  eng.close()


@pytest.mark.parametrize('sampler,weight', [('ddpm', 2.0), ('ddim', 2.0), ('ddpm', 1.0)])
def test_sample_matches_oracle(cuda_device, tiny, sampler, weight):
  t5, params = tiny
  B, steps = 2, 12
  toks, ctx, cmask = H.make_batch(B, T, C)
  init_z, noise = H.make_noise(steps, B, N)
  eng = H.build_engine(t5, T, N, C, B, steps, weight, params, sampler=sampler)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
             b['encoder_continuous_mask'])
  mel = eng.sample(init_z.to(cuda_device), noise.to(cuda_device)).cpu()
  oc = H.oracle_config(t5, steps, weight, sampler=sampler)
  ref, scores = O.predict_batch_with_aux(O.params_to(params), oc, H.torch_batch(toks, ctx, cmask),
                                         init_z, noise)
  span = oc.max_value - oc.min_value
  err = (mel - ref).abs() / span * 2.0     # normalised [-1, 1] units
  assert torch.isfinite(mel).all()
  # tolerance (bf16 operand path, SURVEY §8d): mean |d| <= 3e-2 in normalised units, plus p99 and
  # the share of elements off by more than 0.1
  H.assert_trajectory_close(err, f'tiny {sampler} w={weight}')
  eng.close()


VARIANTS = {
    # name: (engine kwargs, oracle kwargs, cond weight)
    'ddpm_medium': (dict(logvar='medium:0.3'), dict(logvar_type='medium:0.3'), 2.0),
    'ddpm_small': (dict(logvar='small'), dict(logvar_type='small'), 2.0),
    'x0_output': (dict(model_output='x0'), dict(model_output='x0'), 2.0),
    'v_output': (dict(model_output='v'), dict(model_output='v'), 2.0),
    'v_output_ddim_noclip_nocfg': (dict(model_output='v', sampler='ddim', clip_x0=False),
                                   dict(model_output='v', sampler='ddim', clip_x0=False), 1.0),
    'x0_output_nocfg': (dict(model_output='x0'), dict(model_output='x0'), 1.0),
    'linear_schedule': (dict(schedule=('linear', 1e-3, 0.3), train_schedule=('linear', 1e-3, 0.3, 12)),
                        dict(schedule='linear', schedule_start=1e-3, schedule_stop=0.3,
                             train_schedule='linear', train_schedule_start=1e-3,
                             train_schedule_stop=0.3, train_schedule_num_steps=12), 2.0),
    'train_linear_sampler_cosine': (dict(train_schedule=('linear', 1e-4, 0.02, 1000), model_output='x0'),
                                    dict(train_schedule='linear', train_schedule_start=1e-4,
                                         train_schedule_stop=0.02, train_schedule_num_steps=1000,
                                         model_output='x0'), 2.0),
}


@pytest.mark.parametrize('name', sorted(VARIANTS))
def test_sampler_variants_match_oracle(cuda_device, tiny, name):
  """The sampler switches of diffusion_utils.py beyond the shipped gin defaults: logvar_type
  small / medium:<frac> (141-156), model_output x0 / v (301-318), linear schedule (189-199),
  separate train / sampler schedules, each with identical injected noise against the oracle."""
  ekw, okw, weight = VARIANTS[name]
  t5, params = tiny
  B, steps = 2, 12
  toks, ctx, cmask = H.make_batch(B, T, C)
  init_z, noise = H.make_noise(steps, B, N, seed=3)
  eng = H.build_engine(t5, T, N, C, B, steps, weight, params, **ekw)
  oc = H.oracle_config(t5, steps, weight, **okw)
  tab = eng.step_table()
  for i in (steps - 1, steps // 2, 1):
    t = np.float32(i + 1.0) / np.float32(steps)
    s_ = np.float32(i) / np.float32(steps)
    np.testing.assert_allclose(tab[i][6], O.sampler_logsnr(t, oc), rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(tab[i][7], O.sampler_logsnr(s_, oc), rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(tab[i][14], O.train_logsnr(t, oc), rtol=2e-4, atol=2e-5)
    if oc.sampler == 'ddpm':
      one = torch.ones(1)
      d = O.diffusion_reverse(one, one, float(tab[i][7]), float(tab[i][6]), oc.logvar_type)
      np.testing.assert_allclose(tab[i][4], d['std'].item(), rtol=1e-4)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
             b['encoder_continuous_mask'])
  mel = eng.sample(init_z.to(cuda_device), noise.to(cuda_device)).cpu()
  ref, _ = O.predict_batch_with_aux(O.params_to(params), oc, H.torch_batch(toks, ctx, cmask),
                                    init_z, noise)
  span = oc.max_value - oc.min_value
  err = (mel - ref).abs() / span * 2.0
  assert torch.isfinite(mel).all()
  H.assert_trajectory_close(err, f'variant {name}')
  eng.close()


def test_sum_cross_attends_matches_oracle(cuda_device):
  """decoder_cross_attend_style='sum_cross_attends' (network.py:199-216): one attention per
  encoder with its own kernels, each zeroed where its source is fully masked, outputs summed."""
  t5 = config.t5_tiny()
  t5.decoder_cross_attend_style = 'sum_cross_attends'
  params = weights.synthetic_params(t5, T, N, C, seed=5)
  assert 'decoder/layers_0/MultiHeadDotProductAttention_1/key/kernel' in params
  B, steps = 3, 8
  toks, ctx, cmask = H.make_batch(B, T, C, ctx_masks=[1, 0, 1])   # segment 1: context fully masked
  cmask[2, 40:] = 0
  init_z, noise = H.make_noise(steps, B, N, seed=2)
  eng = H.build_engine(t5, T, N, C, B, steps, 2.0, params)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'], b['encoder_continuous_mask'])
  oc = H.oracle_config(t5, steps, 2.0)
  assert oc.decoder_cross_attend_style == 'sum_cross_attends'
  # one conditioned decoder forward ...
  z = init_z.to(cuda_device)
  eps = eng.decode_eps(z, steps - 1, True).cpu()
  p = O.params_to(params)
  cb = H.torch_batch(toks, ctx, cmask)
  encs = O.encode(p, oc, cb['encoder_input_tokens'],
                  O.scale_features(cb['encoder_continuous_inputs'], oc, clip=True),
                  cb['encoder_continuous_mask'])
  want = O.decode(p, oc, encs, init_z, torch.full((B,), 1.0))
  assert _rel(eps, want) < 3e-2
  # ... and the whole trajectory
  mel = eng.sample(z, noise.to(cuda_device)).cpu()
  ref, _ = O.predict_batch_with_aux(p, oc, cb, init_z, noise)
  err = (mel - ref).abs() / (oc.max_value - oc.min_value) * 2.0
  assert torch.isfinite(mel).all()
  H.assert_trajectory_close(err, 'sum_cross_attends')
  eng.close()


def test_tail_split_inside_the_step_graph(cuda_device, monkeypatch):
  """B = 8 base-sized cross-attention (96 CTAs) runs in long/short CTA pairs inside the captured
  step graph; the hand-shake words must re-arm across layers and steps.  Compared with the same
  engine built with the split disabled (same math, different summation order)."""
  t5 = config.t5_small()
  Ts, Ns, Cs, B, steps = 2048, 256, 256, 13, 3          # 13 x 6 heads = 78 CTAs, 18 key blocks
  params = weights.synthetic_params(t5, Ts, Ns, Cs, seed=2)
  toks, ctx, cmask = H.make_batch(B, Ts, Cs, seed=8, pad_second=True)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  outs = []
  monkeypatch.setenv('MSD_ATTN_BKV', '128')   # the tail split belongs to the 128-key instance
  for tail in ('-1', '0'):
    monkeypatch.setenv('MSD_ATTN_TAIL', tail)
    eng = H.build_engine(t5, Ts, Ns, Cs, B, steps, 2.0, params)
    eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
               b['encoder_continuous_mask'])
    outs.append([eng.sample(seed=3).clone(), eng.sample(seed=3).clone()])
    eng.close()
  (plain, plain2), (split, split2) = outs
  assert torch.equal(plain, plain2) and torch.equal(split, split2)       # deterministic, re-armed
  span = 4.0 - np.log(1e-5)
  err = (plain - split).abs() / span * 2.0
  assert torch.isfinite(split).all()
  # random weights saturate most of the 3-step output at the x0 clip, so a rounding-level change
  # (different summation order) flips a few elements across the whole range; bound their share
  assert err.mean().item() < 1e-2, (err.mean().item(), err.max().item())
  assert (err > 0.1).float().mean().item() < 1e-2
  assert not torch.equal(plain, split)                                   # the split really ran


def test_owner_merge_inside_the_step_graph(cuda_device, monkeypatch):
  """64-key instance: a cross-attention whose grid is split along the keys (13 x 6 heads = 78 CTAs
  -> 3 splits = 234 CTAs, one wave of two CTAs per SM) with the owner CTAs merging their partners'
  partials inside the kernel; the flag words must re-arm across layers, steps and calls.  Compared
  with the same engine using the combine kernel (same math, different summation order) and with
  the 128-key instance."""
  t5 = config.t5_small()
  Ts, Ns, Cs, B, steps = 2048, 256, 256, 13, 3
  params = weights.synthetic_params(t5, Ts, Ns, Cs, seed=2)
  toks, ctx, cmask = H.make_batch(B, Ts, Cs, seed=8, pad_second=True)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  outs = {}
  for name, env in (('merge', {'MSD_ATTN_BKV': '64', 'MSD_ATTN_MERGE': '1'}),
                    ('combine', {'MSD_ATTN_BKV': '64', 'MSD_ATTN_MERGE': '0'}),
                    ('bkv128', {'MSD_ATTN_BKV': '128', 'MSD_ATTN_MERGE': '0'})):
    for k, v in env.items():
      monkeypatch.setenv(k, v)
    eng = H.build_engine(t5, Ts, Ns, Cs, B, steps, 2.0, params)
    eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
               b['encoder_continuous_mask'])
    first, second = eng.sample(seed=3).clone(), eng.sample(seed=3).clone()
    assert torch.equal(first, second), name                 # deterministic, flags re-armed
    assert torch.isfinite(first).all(), name
    outs[name] = first
    eng.close()
  span = 4.0 - np.log(1e-5)
  for other in ('combine', 'bkv128'):
    err = (outs['merge'] - outs[other]).abs() / span * 2.0
    assert err.mean().item() < 1e-2, (other, err.mean().item(), err.max().item())
    assert (err > 0.1).float().mean().item() < 1e-2, other


@pytest.mark.parametrize('style', ['concat_encodings', 'sum_cross_attends'])
def test_deferred_normalisation_agrees_with_the_rmsnorm_kernels(cuda_device, monkeypatch, style):
  """bf16 mode folds every pre-norm (+FiLM) of the decoder layers into the GEMM epilogues either
  side of it (DESIGN section 5); MSD_FUSED_NORM=0 keeps the stand-alone rmsnorm kernels.  Same
  math, different rounding points: the two must agree far inside the oracle tolerance, for both
  guidance passes (B = 3: the conditional rows end inside a 256-row tile) and both cross styles."""
  t5 = config.t5_small()
  t5.decoder_cross_attend_style = style
  Ts, Ns, Cs, B, steps = 256, 256, 256, 3, 8
  params = weights.synthetic_params(t5, Ts, Ns, Cs, seed=4)
  toks, ctx, cmask = H.make_batch(B, Ts, Cs, seed=5, pad_second=True)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  z = torch.randn(B, Ns, 128, device=cuda_device, generator=torch.Generator(cuda_device).manual_seed(1))
  outs = {}
  for mode in ('0', '1'):
    monkeypatch.setenv('MSD_FUSED_NORM', mode)
    eng = H.build_engine(t5, Ts, Ns, Cs, B, steps, 2.0, params)
    eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
               b['encoder_continuous_mask'])
    first, second = eng.sample(seed=3).clone(), eng.sample(seed=3).clone()
    assert torch.equal(first, second), mode
    outs[mode] = (eng.decode_eps(z, 5, True).clone(), eng.decode_eps(z, 5, False).clone(), first)
    eng.close()
  for got, want in zip(outs['1'][:2], outs['0'][:2]):
    rel = ((got - want).abs().mean() / want.abs().mean()).item()
    assert rel < 1e-2, rel
  span = 4.0 - np.log(1e-5)
  err = (outs['1'][2] - outs['0'][2]).abs() / span * 2.0
  assert err.mean().item() < 1e-2 and (err > 0.1).float().mean().item() < 1e-2


def test_jax_random_stream_on_device_matches_numpy(cuda_device):
  """rng_kind = 1: the sampler's noise is jax.random.normal of PRNGKey(seed) / fold_in(key, i)
  (inference.py:203; diffusion_utils.py:389-390, 462).  Device draw vs jax_rng.py (numpy), which
  tests/test_jax_rng.py pins on the published vectors."""
  from music_spectrogram_diffusion_b200 import engine, jax_rng as J
  # the values the JAX docs print for PRNGKey(0), straight from the device generator
  got = engine.op_jax_normal(0, -1, 8, cuda_device).cpu().numpy()
  np.testing.assert_allclose(got, J.normal(J.prng_key(0), (8,)), rtol=0, atol=2e-7)
  for seed, step, n in ((0, -1, 32768), (7, 0, 4096), (123456789, 999, 2 * 256 * 128),
                        ((5 << 32) | 77, 3, 8)):
    want = J.init_z(seed, (n,)) if step < 0 else J.step_noise(seed, step, (n,))
    got = engine.op_jax_normal(seed, step, n, cuda_device).cpu().numpy()
    # log1p / sqrt differ from numpy by an ulp or two in the tails
    np.testing.assert_allclose(got, want, rtol=3e-6, atol=3e-7)


def test_seeded_sampling_follows_the_jax_stream(cuda_device, tiny):
  """msd_sample(seed) with rng='jax' == msd_sample with init_z = normal(PRNGKey(seed)) and
  noise[i] = normal(fold_in(key, i)) injected.  The injected draws come from the device generator
  (bit-identical inputs -> bit-identical output; an ulp of difference in a normal is amplified
  22026x by the first reverse step, so numpy-generated draws only agree statistically); the
  generator itself is checked against numpy in the test above."""
  from music_spectrogram_diffusion_b200 import engine
  t5, params = tiny
  B, steps = 2, 6
  toks, ctx, cmask = H.make_batch(B, T, C)
  eng = H.build_engine(t5, T, N, C, B, steps, 2.0, params)
  assert eng.cfg.rng_kind == 1
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'], b['encoder_continuous_mask'])
  shape = (B, N, 128)
  n = B * N * 128
  for seed in (0, 31337, (9 << 32) | 5):
    seeded = eng.sample(seed=seed).clone()
    z0 = engine.op_jax_normal(seed, -1, n, cuda_device).view(shape)
    noise = torch.stack([engine.op_jax_normal(seed, i, n, cuda_device).view(shape) for i in range(steps)])
    injected = eng.sample(z0.contiguous(), noise.contiguous()).clone()
    assert torch.equal(seeded, injected), (seed, (seeded - injected).abs().max().item())
  assert not torch.equal(eng.sample(seed=1), eng.sample(seed=2))
  eng.close()


def test_small_model_one_segment_ten_steps(cuda_device):
  """BASELINE config 0: small model (gin/models/diffusion/context/t5_small.gin), 1 segment of
  256 frames x 128 mel bins, 2048 tokens, 10 DDPM steps, against the CPU oracle."""
  t5 = config.t5_small()
  Ts, Ns, Cs, steps = 2048, 256, 256, 10
  params = weights.synthetic_params(t5, Ts, Ns, Cs, seed=1)
  toks, ctx, cmask = H.make_batch(1, Ts, Cs, seed=4, ctx_masks=[1])
  toks[0, 1500:] = 0                                 # a realistic, padded token segment
  init_z, noise = H.make_noise(steps, 1, Ns, seed=6)
  eng = H.build_engine(t5, Ts, Ns, Cs, 1, steps, 2.0, params)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'], b['encoder_continuous_mask'])
  mel = eng.sample(init_z.to(cuda_device), noise.to(cuda_device)).cpu()
  oc = H.oracle_config(t5, steps, 2.0)
  ref, _ = O.predict_batch_with_aux(O.params_to(params), oc, H.torch_batch(toks, ctx, cmask),
                                    init_z, noise)
  err = (mel - ref).abs() / (oc.max_value - oc.min_value) * 2.0
  assert mel.shape == (1, 256, 128) and torch.isfinite(mel).all()
  H.assert_trajectory_close(err, 'small, 1 segment, 10 steps')
  eng.close()


def test_sample_internal_rng_is_deterministic(cuda_device, tiny):
  t5, params = tiny
  B, steps = 1, 6
  toks, ctx, cmask = H.make_batch(B, T, C)
  eng = H.build_engine(t5, T, N, C, B, steps, 2.0, params)
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'],
             b['encoder_continuous_mask'])
  a = eng.sample(seed=7).clone()
  b2 = eng.sample(seed=7).clone()
  c = eng.sample(seed=8).clone()
  assert torch.equal(a, b2)
  assert not torch.equal(a, c)
  assert torch.isfinite(a).all()
  lo, hi = np.log(1e-5) - 1e-3, 4.0 + 1e-3
  assert a.min().item() >= lo and a.max().item() <= hi
  eng.close()


def test_inference_model_predict_matches_golden_fixture(cuda_device):
  """Through the reference-facing API (host numpy batch in, numpy mel out) against the committed
  fixture tests/golden/tiny_predict.npz (oracle outputs, see make_golden.py)."""
  import os
  from music_spectrogram_diffusion_b200 import inference
  g = H.tiny_golden(os.path.join(os.path.dirname(__file__), 'golden', 'tiny_predict.npz'))
  t5 = config.t5_tiny()
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = int(g['steps'])
  diff.classifier_free_guidance.eval_condition_weight = float(g['cond_weight'])
  lengths = {'inputs': T, 'targets': N, 'targets_context': C}
  model = inference.InferenceModel.from_config(t5, diff, lengths, 'synthetic:0',
                                               batch_size=g['tokens'].shape[0])
  batch = dict(encoder_input_tokens=g['tokens'], encoder_continuous_inputs=g['ctx'],
               encoder_continuous_mask=g['ctx_mask'],
               decoder_target_tokens=np.zeros((g['tokens'].shape[0], N, 128), np.float32))
  mel, scores = model.predict(batch, seed=0, init_z=g['init_z'], noise=g['noise'])
  assert mel.shape == g['mel'].shape and mel.dtype == np.float32
  assert scores.shape == (g['tokens'].shape[0],) and not scores.any()
  span = 4.0 - np.log(1e-5)
  err = np.abs(mel - g['mel']) / span * 2.0
  H.assert_trajectory_close(err, 'tiny golden fixture through InferenceModel.predict')
  with pytest.raises(ValueError):
    model.predict(dict(batch, encoder_input_tokens=g['tokens'][:, :64]))


def test_inference_model_restores_t5x_checkpoint(cuda_device, tiny, tmp_path):
  """InferenceModel(checkpoint_path=<T5X directory>, gin_config) -- the colab's call
  (ipynb:203-229) -- gives bit-identical output to the same tree handed over in memory."""
  import os
  from music_spectrogram_diffusion_b200 import inference, t5x_checkpoint
  t5, params = tiny
  ck = t5x_checkpoint.save_t5x_checkpoint(str(tmp_path / 'checkpoint_500000'), params, step=500000,
                                          inline_below=300, chunk_rows=64)
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = 4
  lengths = {'inputs': T, 'targets': N, 'targets_context': C}
  a = inference.InferenceModel.from_config(t5, diff, lengths, ck, 1)
  b = inference.InferenceModel.from_config(t5, diff, lengths, 'synthetic:0', 1, params=params)
  rng = np.random.default_rng(9)
  batch = dict(encoder_input_tokens=rng.integers(3, 1391, (1, T)).astype(np.int32),
               encoder_continuous_inputs=rng.uniform(-11, 4, (1, C, 128)).astype(np.float32),
               encoder_continuous_mask=np.ones((1, C), np.int32),
               decoder_target_tokens=np.zeros((1, N, 128), np.float32))
  ma, _ = a.predict(batch, seed=3)
  mb, _ = b.predict(batch, seed=3)
  np.testing.assert_array_equal(ma, mb)
  with pytest.raises(ValueError, match='does not match the gin config'):
    inference.InferenceModel.from_config(config.t5_small(), diff, lengths, ck, 1).predict(batch)


def test_song_driver_end_to_end(cuda_device, tiny):
  """song.synthesize_song (notes -> tokens -> chained predict) on the real engine equals the
  same chain driven by hand through InferenceModel.predict."""
  from music_spectrogram_diffusion_b200 import inference, midi_tokens as M, song
  t5, params = tiny
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = 5
  diff.classifier_free_guidance.eval_condition_weight = 2.0
  lengths = {'inputs': T, 'targets': N, 'targets_context': C}
  model = inference.InferenceModel.from_config(t5, diff, lengths, 'synthetic:0', 1, params=params)
  notes = M.make_notes([(0.2, 4.0, 60, 100, 0, False), (1.0, 1.3, 38, 110, 0, True),
                        (3.0, 3.4, 67, 80, 41, False)])
  out = song.synthesize_song(model, notes, seed=4)
  nseg = -(-M.num_song_frames(4.0) // N)
  assert nseg == 2 and out['full_pred_encoded'].shape == (nseg * N, 128)
  assert np.isfinite(out['full_pred_encoded']).all()
  assert out['model_timing']['prediction_seconds_per_chunk'] > 0
  prev = np.zeros((1, C, 128), np.float32)
  for i in range(nseg):
    batch = dict(encoder_input_tokens=out['tokens'][i:i + 1], encoder_continuous_inputs=prev,
                 encoder_continuous_mask=np.full((1, C), 0 if i == 0 else 1, np.int32),
                 decoder_target_tokens=np.zeros((1, N, 128), np.float32))
    prev, _ = model.predict(batch, seed=4)
    np.testing.assert_array_equal(out['full_pred_encoded'][i * N:(i + 1) * N], prev[0])


def test_chained_song_single_gpu(cuda_device, tiny):
  """distributed.synthesize_song on one rank == the colab loop (ipynb:895-935): first segment
  masked context, later ones fed the previous prediction."""
  from music_spectrogram_diffusion_b200 import distributed as D, inference
  t5, params = tiny
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = 6
  diff.classifier_free_guidance.eval_condition_weight = 2.0
  lengths = {'inputs': T, 'targets': N, 'targets_context': C}
  model = inference.InferenceModel.from_config(t5, diff, lengths, 'synthetic:0', 1, params=params)
  rng = np.random.default_rng(4)
  segs = [torch.from_numpy(rng.integers(3, 1391, (T,)).astype(np.int32)) for _ in range(3)]
  song = D.synthesize_song(model.predict_on_device, segs, C, 128, cuda_device, seed=5)
  assert song.shape == (1, 3 * N, 128) and torch.isfinite(song).all()
  # manual loop through the host API
  prev = np.zeros((1, C, 128), np.float32)
  outs = []
  for k, s in enumerate(segs):
    b = dict(encoder_input_tokens=s.numpy()[None], encoder_continuous_inputs=prev,
             encoder_continuous_mask=np.full((1, C), 0 if k == 0 else 1, np.int32))
    prev, _ = model.predict(b, seed=5)
    outs.append(prev)
  np.testing.assert_array_equal(song.cpu().numpy(), np.concatenate(outs, axis=1))


@pytest.mark.parametrize('steps', [20, 1000])
def test_base_with_context_matches_oracle_fixture(cuda_device, steps):
  """BASELINE config 2: base_with_context, 1 segment, CFG 2.0, fp32 oracle (graph as written) vs
  the CUDA path, both driven by the library's Philox noise from the same seed.  Fixture:
  tests/golden/base_predict_<steps>.npz (tests/golden/make_base_golden.py; the 1000-step one costs
  ~20 CPU-minutes)."""
  import os
  import bench
  from music_spectrogram_diffusion_b200 import inference
  path = os.path.join(os.path.dirname(__file__), 'golden', f'base_predict_{steps}.npz')
  if not os.path.exists(path):
    pytest.skip(f'{os.path.basename(path)} not generated')
  g = np.load(path)
  t5 = config.t5_base()
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = int(g['steps'])
  diff.classifier_free_guidance.eval_condition_weight = float(g['cond_weight'])
  lengths = dict(config.TASK_FEATURE_LENGTHS_CONTEXT)
  model = inference.InferenceModel.from_config(t5, diff, lengths,
                                               f'synthetic:{int(g["weight_seed"])}', batch_size=1,
                                               rng='philox')
  batch = bench.synthetic_batch(1, lengths, seed=int(g['batch_seed']))
  mel, _ = model.predict(batch, seed=int(g['seed']))
  span = 4.0 - np.log(1e-5)
  err = np.abs(mel - g['mel']) / span * 2.0
  assert np.isfinite(mel).all()
  H.assert_trajectory_close(err, f'base_with_context, 1 segment, {steps} steps')


def test_base_with_context_batch8_matches_oracle_fixture(cuda_device):
  """BASELINE config 3 -- the configuration bench.py measures: base_with_context, batch of 8
  segments through InferenceModel.predict(batch_size=8) (256-wide CTA-pair GEMM tiles at M = 4096,
  the long/short cross-attention split inside the captured step graph), mixed token padding, one
  fully masked and one partially filled context, against the fp32 oracle (graph as written).
  Fixture: tests/golden/base_b8_predict_20.npz (tests/golden/make_base_b8_golden.py)."""
  import os
  from music_spectrogram_diffusion_b200 import inference
  path = os.path.join(os.path.dirname(__file__), 'golden', 'base_b8_predict_20.npz')
  g = np.load(path)
  t5 = config.t5_base()
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = int(g['steps'])
  diff.classifier_free_guidance.eval_condition_weight = float(g['cond_weight'])
  lengths = dict(config.TASK_FEATURE_LENGTHS_CONTEXT)
  model = inference.InferenceModel.from_config(t5, diff, lengths,
                                               f'synthetic:{int(g["weight_seed"])}', batch_size=8,
                                               rng='philox')
  batch = H.base_b8_batch(lengths, int(g['batch_seed']))
  mel, _ = model.predict(batch, seed=int(g['seed']))
  assert mel.shape == (8, 256, 128) and np.isfinite(mel).all()
  span = 4.0 - np.log(1e-5)
  err = np.abs(mel - g['mel']) / span * 2.0
  H.assert_trajectory_close(err, 'base_with_context, 8 segments, 20 steps')
  for seg in range(8):   # no segment hides behind the batch average
    H.assert_trajectory_close(err[seg], f'  segment {seg}')


# ---- fp32-accurate mode (BASELINE config 2) ------------------------------------------------------
def test_fp32_accurate_decoder_forward(cuda_device, tiny):
  """precision='fp32_accurate': one decoder forward (network.py:360-457) to ~1e-4 of the fp32
  oracle (SURVEY 8d: max|d eps| <= 1e-4 rms for the fp32-accurate path; the 3 x bf16 split keeps
  ~16 mantissa bits per operand), conditioned and unconditioned, plus the encoders."""
  t5, params = tiny
  B, steps = 3, 16
  toks, ctx, cmask = H.make_batch(B, T, C, ctx_masks=[1, 0, 1])
  cmask[2, 40:] = 0
  eng = H.build_engine(t5, T, N, C, B, steps, 2.0, params, precision='fp32_accurate')
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'], b['encoder_continuous_mask'])
  oc = H.oracle_config(t5, steps, 2.0)
  P = O.params_to(params)
  cb = H.torch_batch(toks, ctx, cmask)
  encs = O.encode(P, oc, cb['encoder_input_tokens'],
                  O.scale_features(cb['encoder_continuous_inputs'], oc, clip=True),
                  cb['encoder_continuous_mask'])
  want = torch.cat([encs[0][0], encs[1][0]], dim=1)
  valid = torch.cat([encs[0][1], encs[1][1]], dim=1) > 0
  err = ((eng.encodings().cpu() - want).abs() * valid.unsqueeze(-1)).max().item()
  assert err < 2e-3, f'encodings: {err}'          # stored as hi + lo: 16 mantissa bits of O(10) values
  z = torch.randn(B, N, 128, generator=torch.Generator().manual_seed(3))
  for conditioned in (True, False):
    flag = 1.0 if conditioned else 0.0
    for step_i in (steps - 1, 5, 0):
      got = eng.decode_eps(z.to(cuda_device), step_i, conditioned).cpu()
      t = np.float32(step_i + 1.0) / np.float32(steps)
      ref = O.decode(P, oc, [(e * flag, m * flag) for e, m in encs], z, torch.full((B,), float(t)))
      rel = ((got - ref).abs().max() / ref.pow(2).mean().sqrt()).item()
      assert rel < 2e-3, f'cond={conditioned} step {step_i}: {rel}'
  eng.close()


@pytest.mark.parametrize('sampler,weight,style', [('ddpm', 2.0, 'concat_encodings'),
                                                   ('ddim', 2.0, 'concat_encodings'),
                                                   ('ddpm', 1.0, 'concat_encodings'),
                                                   ('ddpm', 2.0, 'sum_cross_attends')])
def test_fp32_accurate_sample_matches_oracle(cuda_device, sampler, weight, style):
  """Full trajectories in the fp32-accurate mode.  SURVEY 8d's fp32 tolerance is mean |d| <= 1e-3
  normalised; measured on B200: mean 3-5e-6, p99 5e-5, max 3e-4 -- the bounds asserted are ten
  times the measured values, i.e. 10x inside the stated tolerance."""
  t5 = config.t5_tiny()
  t5.decoder_cross_attend_style = style
  params = weights.synthetic_params(t5, T, N, C, seed=0 if style == 'concat_encodings' else 5)
  B, steps = 2, 12
  toks, ctx, cmask = H.make_batch(B, T, C)
  init_z, noise = H.make_noise(steps, B, N)
  eng = H.build_engine(t5, T, N, C, B, steps, weight, params, sampler=sampler,
                       precision='fp32_accurate')
  b = H.torch_batch(toks, ctx, cmask, cuda_device)
  eng.encode(b['encoder_input_tokens'], b['encoder_continuous_inputs'], b['encoder_continuous_mask'])
  mel = eng.sample(init_z.to(cuda_device), noise.to(cuda_device)).cpu()
  oc = H.oracle_config(t5, steps, weight, sampler=sampler)
  ref, _ = O.predict_batch_with_aux(O.params_to(params), oc, H.torch_batch(toks, ctx, cmask),
                                    init_z, noise)
  err = (mel - ref).abs() / (oc.max_value - oc.min_value) * 2.0
  H.assert_trajectory_close(err, f'fp32-accurate tiny {sampler} w={weight} {style}',
                            mean=1e-4, p99=1e-3, share_01=1e-5)
  eng.close()


@pytest.mark.parametrize('steps', [20, 1000])
def test_fp32_accurate_base_with_context_matches_oracle_fixture(cuda_device, steps):
  """BASELINE config 2 as written: base_with_context, 1 segment, fp32 vs the reference tolerance
  (SURVEY 8d: mean |d| <= 1e-3 normalised over the full trajectory).  Measured on B200 at 20
  steps: mean 1.0e-5, p99 1.3e-4, max 6e-4; asserted: 10x those, still 10x inside 1e-3."""
  import os
  import bench
  from music_spectrogram_diffusion_b200 import inference
  g = np.load(os.path.join(os.path.dirname(__file__), 'golden', f'base_predict_{steps}.npz'))
  t5 = config.t5_base()
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = int(g['steps'])
  diff.classifier_free_guidance.eval_condition_weight = float(g['cond_weight'])
  lengths = dict(config.TASK_FEATURE_LENGTHS_CONTEXT)
  model = inference.InferenceModel.from_config(
      t5, diff, lengths, f'synthetic:{int(g["weight_seed"])}', batch_size=1, rng='philox',
      precision='fp32_accurate')
  batch = bench.synthetic_batch(1, lengths, seed=int(g['batch_seed']))
  # the very draws the fixture was made with (oracle/philox.py, numpy), injected: the device
  # generator agrees with numpy only to an ulp or two (sincospif vs float64 cos), which this
  # tolerance would see
  from oracle import philox
  shape, seed = (1, 256, 128), int(g['seed'])
  init_z = philox.init_z(seed, shape)
  noise = np.stack([philox.step_noise(seed, i, shape) for i in range(steps)])
  mel, _ = model.predict(batch, seed=seed, init_z=init_z, noise=noise)
  err = np.abs(mel - g['mel']) / (4.0 - np.log(1e-5)) * 2.0
  assert np.isfinite(mel).all()
  H.assert_trajectory_close(err, f'fp32-accurate base_with_context, 1 segment, {steps} steps',
                            mean=1e-4, p99=1.5e-3, share_01=1e-5)
