"""CPU: structural properties of the oracle restatement that the CUDA path relies on -- the
exact algebraic shortcuts (hoisted cross K/V is implicit; elided unconditional cross-attention;
tabulated FiLM), fp32-vs-fp64 self-consistency, and the committed golden fixture."""
import os

import numpy as np
import pytest
import torch

from music_spectrogram_diffusion_b200 import config, weights
from oracle import msd_oracle as O
from tests import helpers as H

T = N = C = 128
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'tiny_predict.npz')


@pytest.fixture(scope='module')
def tiny():
  t5 = config.t5_tiny()
  params = weights.synthetic_params(t5, T, N, C, seed=0)
  return t5, params


def _decoder_without_cross(P, oc, z, time):
  """Decoder with the cross-attention branch removed entirely."""
  c = O.conditioning_embedding(time, P, oc)
  y = O.dense_general(z, P['decoder/continuous_inputs_projection/kernel'])
  y = y + P['decoder/Embed_0/embedding'][:z.shape[1]][None]
  for l in range(oc.num_decoder_layers):
    p = f'decoder/layers_{l}'
    x = O.layer_norm(y, P[f'{p}/pre_self_attention_layer_norm/scale'])
    x = O.film_layer(x, c, P[f'{p}/FiLMLayer_0/DenseGeneral_0/kernel'])
    x = O.multi_head_dot_product_attention(x, x, None, P, f'{p}/self_attention', oc.num_heads,
                                           oc.head_dim) + y
    v = O.layer_norm(x, P[f'{p}/pre_mlp_layer_norm/scale'])
    v = O.film_layer(v, c, P[f'{p}/FiLMLayer_1/DenseGeneral_0/kernel'])
    y = O.mlp_block(v, P, f'{p}/mlp', oc.mlp_activations) + x
  y = O.layer_norm(y, P['decoder/decoder_norm/scale'])
  return O.dense_general(y, P['decoder/spec_out_dense/kernel'])


def test_unconditional_pass_has_exactly_zero_cross_attention(tiny):
  """models.py:376-377 multiplies encodings AND masks by 0 -> zero_activations_if_masked makes
  the cross-attention branch exactly 0, so the CUDA path may skip it (bit-for-bit)."""
  t5, params = tiny
  oc = H.oracle_config(t5, 8, 2.0)
  P = O.params_to(params)
  toks, ctx, cmask = H.make_batch(2, T, C)
  b = H.torch_batch(toks, ctx, cmask)
  encs = O.encode(P, oc, b['encoder_input_tokens'],
                  O.scale_features(b['encoder_continuous_inputs'], oc, clip=True),
                  b['encoder_continuous_mask'])
  z = torch.randn(2, N, 128, generator=torch.Generator().manual_seed(5))
  time = torch.full((2,), 0.375)
  as_written = O.decode(P, oc, [(e * 0.0, m * 0.0) for e, m in encs], z, time)
  skipped = _decoder_without_cross(P, oc, z, time)
  assert torch.equal(as_written, skipped)


def test_film_depends_only_on_step_index(tiny):
  """network.py:377-394: the conditioning embedding is a function of `time` alone, identical for
  every batch row -> it can be tabulated per step at load time."""
  t5, params = tiny
  oc = H.oracle_config(t5, 16, 2.0)
  P = O.params_to(params)
  for i in (0, 7, 15):
    t = np.float32(i + 1.0) / np.float32(16)
    c = O.conditioning_embedding(torch.full((3,), float(t)), P, oc)
    assert torch.equal(c[0], c[1]) and torch.equal(c[0], c[2])
    sb = O.dense_general(c, P['decoder/layers_0/FiLMLayer_0/DenseGeneral_0/kernel'])
    assert sb.shape == (3, 1, 2 * t5.emb_dim)


def test_fully_masked_context_does_not_influence_output(tiny):
  """First-segment case: ctx mask all zero -> the context encodings are masked keys in every
  cross-attention; their values (which come from a uniform-softmax encoder pass) are irrelevant."""
  t5, params = tiny
  oc = H.oracle_config(t5, 4, 2.0)
  P = O.params_to(params)
  toks, ctx, cmask = H.make_batch(1, T, C, ctx_masks=[0])
  b = H.torch_batch(toks, ctx, cmask)
  z = torch.randn(1, N, 128, generator=torch.Generator().manual_seed(6))
  time = torch.full((1,), 0.5)
  outs = []
  for scale in (1.0, -3.0):
    encs = O.encode(P, oc, b['encoder_input_tokens'],
                    O.scale_features(b['encoder_continuous_inputs'] * scale, oc, clip=True),
                    b['encoder_continuous_mask'])
    outs.append(O.decode(P, oc, encs, z, time))
  assert torch.allclose(outs[0], outs[1], atol=0, rtol=0)


def test_fp32_oracle_tracks_fp64(tiny):
  t5, params = tiny
  steps = 10
  oc = H.oracle_config(t5, steps, 2.0)
  toks, ctx, cmask = H.make_batch(2, T, C)
  init_z, noise = H.make_noise(steps, 2, N)
  b = H.torch_batch(toks, ctx, cmask)
  mel32, _ = O.predict_batch_with_aux(O.params_to(params), oc, b, init_z, noise)
  mel64, _ = O.predict_batch_with_aux(O.params_to(params, torch.float64), oc, b, init_z.double(),
                                      noise.double())
  span = oc.max_value - oc.min_value
  err = (mel32.double() - mel64).abs() / span * 2
  assert err.mean().item() < 1e-4 and err.max().item() < 5e-3


def test_last_step_returns_clipped_x0_without_noise(tiny):
  """diffusion_utils.py:395: i == 0 returns pred_x0 (clipped), ignoring the noise."""
  t5, _ = tiny
  oc = H.oracle_config(t5, 4, 2.0)
  z = torch.randn(1, 4, 128)
  pred = lambda zz, t, c: torch.full_like(zz, 0.3 if c else -0.1)
  a = O.eval_step(z, 0, torch.zeros_like(z), pred, oc)
  b = O.eval_step(z, 0, torch.full_like(z, 1e6), pred, oc)
  assert torch.equal(a, b) and a.abs().max() <= 1.0


def test_golden_fixture_matches_live_oracle(tiny):
  """tests/golden/tiny_predict.npz (written by tests/golden/make_golden.py) pins today's oracle
  output so an accidental change of the restatement is caught."""
  t5, params = tiny
  g = H.tiny_golden(GOLDEN)
  steps = int(g['steps'])
  oc = H.oracle_config(t5, steps, float(g['cond_weight']))
  batch = dict(encoder_input_tokens=torch.from_numpy(g['tokens']),
               encoder_continuous_inputs=torch.from_numpy(g['ctx']),
               encoder_continuous_mask=torch.from_numpy(g['ctx_mask']))
  mel, _ = O.predict_batch_with_aux(O.params_to(params), oc, batch, torch.from_numpy(g['init_z']),
                                    torch.from_numpy(g['noise']))
  np.testing.assert_allclose(mel.numpy(), g['mel'], atol=2e-3)
  eps = O.decode(O.params_to(params), oc,
                 O.encode(O.params_to(params), oc, batch['encoder_input_tokens'],
                          O.scale_features(batch['encoder_continuous_inputs'], oc, clip=True),
                          batch['encoder_continuous_mask']),
                 torch.from_numpy(g['init_z']), torch.full((g['init_z'].shape[0],), 1.0))
  np.testing.assert_allclose(eps.numpy(), g['eps_first'], atol=2e-4)
