"""Writes tests/golden/tiny_predict.npz: seeded inputs and the ORACLE's outputs for the tiny
network (config.t5_tiny, synthetic_params seed 0).  The reference itself cannot be imported in
this image (no jax/flax/t5x), so these vectors pin the oracle restatement, not the reference;
see oracle/msd_oracle.py "PARITY STATUS".  Run from the repo root: python tests/golden/make_golden.py"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from music_spectrogram_diffusion_b200 import config, weights  # noqa: E402
from oracle import msd_oracle as O  # noqa: E402
from tests import helpers as H  # noqa: E402

T = N = C = 128
STEPS, W, B, NOISE_SEED = 12, 2.0, 2, 0
t5 = config.t5_tiny()
params = weights.synthetic_params(t5, T, N, C, seed=0)
toks, ctx, cmask = H.make_batch(B, T, C)
init_z, noise = H.make_noise(STEPS, B, N, seed=NOISE_SEED)
oc = H.oracle_config(t5, STEPS, W)
P = O.params_to(params)
batch = H.torch_batch(toks, ctx, cmask)
mel, _ = O.predict_batch_with_aux(P, oc, batch, init_z, noise)
encs = O.encode(P, oc, batch['encoder_input_tokens'],
                O.scale_features(batch['encoder_continuous_inputs'], oc, clip=True),
                batch['encoder_continuous_mask'])
eps_first = O.decode(P, oc, encs, init_z, torch.full((B,), 1.0))
# the noise itself is redrawn from NOISE_SEED by tests/helpers.tiny_golden; a sample pins it
np.savez_compressed(
    os.path.join(os.path.dirname(os.path.abspath(__file__)), 'tiny_predict.npz'),
    tokens=toks, ctx=ctx, ctx_mask=cmask, init_z=init_z.numpy(), noise_seed=NOISE_SEED,
    noise_sample=noise[:, :, 0, :8].numpy(), mel=mel.numpy(), eps_first=eps_first.numpy(),
    steps=STEPS, cond_weight=W)
print('wrote tiny_predict.npz', mel.shape, float(mel.mean()))
