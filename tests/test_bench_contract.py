"""bench.py contract pieces that run without a GPU: the reference arm's JSON line, the
rank-0-only rule under torchrun, and the algorithmic FLOP model behind `roofline` / `whole_step`
(SURVEY App. C)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from music_spectrogram_diffusion_b200 import config  # noqa: E402


def _run(extra_env=None):
  env = dict(os.environ)
  env.pop('RANK', None)
  env.pop('WORLD_SIZE', None)
  env.update(extra_env or {})
  return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference',
                         '--model', 'tiny', '--steps', '1', '--warmup', '0', '--diffusion-steps', '4'],
                        env=env, cwd=ROOT, capture_output=True, text=True, timeout=300)


def test_reference_arm_prints_one_contract_line():
  out = _run()
  assert out.returncode == 0, out.stderr[-500:]
  lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
  assert len(lines) == 1
  j = json.loads(lines[0])
  assert j['impl'] == 'reference' and j['metric'] == 'mel-frames/sec' and j['unit'] == 'frames/s'
  assert j['higher_is_better'] is True and j['scaling'] == 'weak' and j['vs_baseline'] is None
  assert j['n_gpus'] == 1 and j['steps'] == 1 and j['warmup'] == 0 and j['value'] > 0
  assert 'workload' in j['config'] and 'model' not in j['config']
  cb = j['cpu_baseline']
  assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == j['value'] and cb['sample']
  assert j['e2e'] == {'value': j['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0,
                      'd2h_bytes_per_step': 0}


def test_reference_arm_runs_on_rank_zero_only():
  out = _run({'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
  assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith('{')]


def test_dump_outputs_writes_float32_within_budget(tmp_path):
  import numpy as np
  import torch
  mel = torch.arange(10 * 4 * 3, dtype=torch.float32).reshape(10, 4, 3)
  bench.dump_outputs(str(tmp_path / 'all'), 'mel', mel)
  got = np.load(tmp_path / 'all' / 'mel.npy')
  assert got.dtype == np.float32 and np.array_equal(got, mel.numpy())
  assert sorted(os.listdir(tmp_path / 'all')) == ['mel.npy']
  # room for 3 segments of 48 bytes (+ 8 index bytes each): a fixed sample of whole segments
  for d in ('a', 'b'):
    bench.dump_outputs(str(tmp_path / d), 'mel', mel, budget=3 * 56)
  idx = np.load(tmp_path / 'a' / 'mel_segments.npy')
  assert idx.dtype == np.float64 and len(idx) == 3 and np.all(np.diff(idx) > 0)
  np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'mel.npy'), mel.numpy()[idx.astype(int)])
  np.testing.assert_array_equal(idx, np.load(tmp_path / 'b' / 'mel_segments.npy'))


def test_bench_refuses_zero_steps_and_reference_dumps(tmp_path):
  for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', str(tmp_path)]):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, cwd=ROOT,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and not out.stdout, out.stderr[-500:]


@pytest.mark.gpu
def test_dumped_outputs_are_what_the_timed_path_computed(tmp_path, cuda_device):
  """--dump-outputs writes the mel of the last timed step: the same bits as InferenceModel.predict
  on the benchmark's seeded batch, and the same in a second run."""
  import numpy as np
  from music_spectrogram_diffusion_b200 import inference
  args = ['--model', 'tiny', '--segments', '2', '--diffusion-steps', '4', '--steps', '2',
          '--warmup', '1', '--no-song', '--no-timeline', '--no-traffic', '--no-cpu-baseline']
  dumps = []
  for run in ('a', 'b'):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args +
                         ['--dump-outputs', str(tmp_path / run)], cwd=ROOT, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert os.listdir(tmp_path / run) == ['mel.npy']
    dumps.append(np.load(tmp_path / run / 'mel.npy'))
  assert dumps[0].dtype == np.float32 and dumps[0].shape == (2, 128, 128)
  np.testing.assert_array_equal(dumps[0], dumps[1])
  t5 = config.t5_tiny()
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = 4
  diff.classifier_free_guidance.eval_condition_weight = 2.0
  lengths = {'inputs': 128, 'targets': 128, 'targets_context': 128}
  model = inference.InferenceModel.from_config(t5, diff, lengths, 'synthetic:0', batch_size=2)
  mel, _ = model.predict(bench.synthetic_batch(2, lengths, seed=100), seed=0)
  np.testing.assert_array_equal(dumps[0], mel)


def test_flop_model_matches_the_survey_derivation():
  lengths = dict(config.TASK_FEATURE_LENGTHS_CONTEXT)
  per_step, once = bench.flops_model(config.t5_base(), lengths)
  assert abs(per_step / 1e9 - 120.997) < 0.01          # cond 74.994 + uncond 46.003 GF per segment
  assert abs(once / 1e9 - 613.7) < 0.2                 # encoders + hoisted cross K/V
  assert abs((per_step * 1000 + once) / 256 / 1e9 - 475.04) < 0.05   # GFLOP per mel frame
  assert abs(bench.as_written_flops(config.t5_base(), lengths) / 1e9 - 280.9) < 0.2
  small, _ = bench.flops_model(config.t5_small(), lengths)
  assert abs(small / 1e9 - 29.93) < 0.05
