"""Shared builders for the parity tests (tiny network + seeded inputs)."""
import numpy as np
import torch

from music_spectrogram_diffusion_b200 import config, engine, weights
from oracle import msd_oracle as O


def bf16_round(t: torch.Tensor) -> torch.Tensor:
  return t.to(torch.bfloat16).to(torch.float32)


def oracle_config(t5, steps, cond_weight, **kw):
  return O.OracleConfig(
      vocab_size=t5.vocab_size, emb_dim=t5.emb_dim, num_heads=t5.num_heads,
      num_encoder_layers=t5.num_encoder_layers, num_decoder_layers=t5.num_decoder_layers,
      head_dim=t5.head_dim, mlp_dim=t5.mlp_dim, num_steps=steps,
      decoder_cross_attend_style=t5.decoder_cross_attend_style,
      eval_condition_weight=cond_weight, **kw)


def make_batch(B, T, C, seed=1, pad_second=True, ctx_masks=None):
  rng = np.random.default_rng(seed)
  toks = rng.integers(3, 1391, (B, T)).astype(np.int32)
  toks[:, -1] = 1
  if pad_second and B > 1:
    toks[1, T // 2 - 4:] = 0
  ctx = rng.uniform(np.log(1e-5) - 1.0, 4.5, (B, C, 128)).astype(np.float32)
  if ctx_masks is None:
    ctx_masks = [1 if i % 2 == 0 else 0 for i in range(B)]
  cmask = np.stack([np.full(C, m, np.int32) for m in ctx_masks])
  return toks, ctx, cmask


def make_noise(steps, B, N, seed=0):
  g = torch.Generator().manual_seed(seed)
  init_z = torch.randn(B, N, 128, generator=g)
  noise = torch.randn(steps, B, N, 128, generator=g)
  return init_z, noise


def tiny_golden(path):
  """tests/golden/tiny_predict.npz (tests/golden/make_golden.py) as a dict.  The per-step noise
  (1.6 MB of incompressible floats) is not stored: it is redrawn by make_noise from the stored
  seed, and the stored init_z and noise sample fail the load if that stream ever changes."""
  g = dict(np.load(path))
  init_z, noise = make_noise(int(g['steps']), g['init_z'].shape[0], g['init_z'].shape[1],
                             seed=int(g['noise_seed']))
  np.testing.assert_array_equal(init_z.numpy(), g['init_z'])
  np.testing.assert_array_equal(noise[:, :, 0, :8].numpy(), g['noise_sample'])
  g['noise'] = noise.numpy()
  return g


def build_engine(t5, T, N, C, B, steps, cond_weight, params, sampler='ddpm', logvar='large',
                 clip_x0=True, model_output='eps', schedule=None, train_schedule=None,
                 precision='bf16'):
  """schedule / train_schedule: None (cosine) or ('linear', start, stop[, num_steps])."""
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = steps
  diff.sampler.name = sampler
  diff.sampler.logvar_type = logvar
  diff.sampler.clip_x0 = clip_x0
  diff.model_output = model_output
  if schedule is not None:
    diff.sampler.schedule = config.DiffusionSchedule(schedule[0], schedule[1], schedule[2], steps)
  if train_schedule is not None:
    diff.train_schedule = config.DiffusionSchedule(*train_schedule)
  diff.classifier_free_guidance.eval_condition_weight = cond_weight
  eng = engine.Engine(engine.make_msd_config(t5, diff, T, N, C, max_batch=B, precision=precision), 0)
  eng.load_weights(params)
  return eng


def torch_batch(toks, ctx, cmask, device=None):
  d = dict(encoder_input_tokens=torch.from_numpy(toks),
           encoder_continuous_inputs=torch.from_numpy(ctx),
           encoder_continuous_mask=torch.from_numpy(cmask))
  if device is not None:
    d = {k: v.to(device) for k, v in d.items()}
  return d


def base_b8_batch(lengths, seed=321):
  """The batch of tests/golden/base_b8_predict_<steps>.npz (BASELINE config 3's shape): 8 segments
  of base_with_context with mixed token padding (full, three padded lengths incl. a nearly empty
  one), out-of-range context values (exercise the clip), one segment with a fully masked context
  (a song's first segment) and one with a partially filled context (terminal-relative roll)."""
  rng = np.random.default_rng(seed)
  T, C = lengths['inputs'], lengths['targets_context']
  toks = rng.integers(3, 1391, (8, T)).astype(np.int32)
  toks[:, -1] = 1
  for seg, n in ((1, 1500), (3, 700), (6, 40)):
    toks[seg, n:] = 0
    toks[seg, n - 1] = 1
  ctx = rng.uniform(np.log(1e-5) - 1.0, 4.5, (8, C, 128)).astype(np.float32)
  cmask = np.ones((8, C), np.int32)
  cmask[2, :] = 0
  cmask[5, 100:] = 0
  return dict(encoder_input_tokens=toks, encoder_continuous_inputs=ctx,
              encoder_continuous_mask=cmask,
              decoder_target_tokens=np.zeros((8, lengths['targets'], 128), np.float32))


def trajectory_stats(err):
  """err: |got - want| in normalised [-1, 1] units (torch or numpy)."""
  e = np.asarray(err.detach().cpu().numpy() if isinstance(err, torch.Tensor) else err, np.float64)
  return dict(mean=float(e.mean()), p99=float(np.quantile(e, 0.99)), max=float(e.max()),
              share_01=float((e > 0.1).mean()))


def assert_trajectory_close(err, what, mean=3e-2, p99=0.12, share_01=0.02):
  """Tolerance of a full sampled trajectory on the bf16-operand path against the fp32 oracle
  (SURVEY 8d), normalised units.  mean: the stated tolerance.  p99 / share of elements off by more
  than 0.1: twice the values measured on base_with_context over 1000 steps (p99 5.8e-2; share
  0.4 %).  Individual elements may flip across the x0 clip (diffusion_utils.py:440-441), so the
  maximum is reported, not bounded."""
  s = trajectory_stats(err)
  print(f'{what}: mean|d|={s["mean"]:.3e} p99={s["p99"]:.3e} share(>0.1)={s["share_01"]:.3e} '
        f'max={s["max"]:.3e}')
  assert np.isfinite(s['max']), what
  assert s['mean'] < mean, (what, s)
  assert s['p99'] < p99, (what, s)
  assert s['share_01'] < share_01, (what, s)
  return s
