"""Writes tests/golden/reference_gin_model_sizes.json: the network.T5Config sizes that gin_lite
reads from the original project's gin/models/diffusion/context/*.gin files.  It first checks that
gin_lite parses every .gin file of that project.  tests/test_host.py compares the stored sizes with
config.py, so the original checkout is only needed to regenerate the file:

    python tests/golden/make_reference_gin_sizes.py --reference /path/to/music-spectrogram-diffusion
"""
import argparse
import glob
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from music_spectrogram_diffusion_b200 import gin_lite  # noqa: E402

MODELS = ('local_tiny', 't5_small', 't5_base', 't5_large')
FIELDS = ('emb_dim', 'num_heads', 'num_decoder_layers', 'mlp_dim')

ap = argparse.ArgumentParser()
ap.add_argument('--reference', required=True, help='checkout of music-spectrogram-diffusion')
args = ap.parse_args()
gin_dir = os.path.join(args.reference, 'music_spectrogram_diffusion', 'gin')
files = sorted(glob.glob(os.path.join(gin_dir, '**', '*.gin'), recursive=True))
assert len(files) >= 25, files
for f in files:
  with open(f) as fh:
    gin_lite.parse_config(fh.read(), [args.reference])
sizes = {}
for name in MODELS:
  with open(os.path.join(gin_dir, 'models', 'diffusion', 'context', name + '.gin')) as fh:
    g = gin_lite.parse_config(fh.read(), [args.reference])
  b = g.bindings_for('network.T5Config')
  sizes[name] = {k: g.resolve(b[k]) for k in FIELDS}
out = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'reference_gin_model_sizes.json')
with open(out, 'w') as fh:
  json.dump(sizes, fh, indent=1)
  fh.write('\n')
print(f'parsed {len(files)} gin files; wrote {out}')
