#!/usr/bin/env python
"""Benchmark of the DDPM sampling hot path (BASELINE.json metric: mel-frames/sec,
base_with_context, 1000-step DDPM).

  python bench.py --gpus N --steps K --warmup W        # this repo's sm_100a path
  python bench.py --impl reference ...                 # the CPU oracle port on the host cores
  python bench.py ... --dump-outputs DIR               # + the last timed step's mel in DIR/mel.npy

A "step" is one pass of the hot path over one batch: `predict` of `--segments` independent
5.12 s segments per GPU (encode + num_steps reverse-diffusion steps + unscale).  Under torchrun
every rank runs the same per-GPU workload (weak scaling, no data-path collective); timing is
barrier + synchronize on both sides, CUDA events on the device, max over ranks.
"""

from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME_RATE = 50.0  # 16000 / 320, msd/audio_codecs.py:162-164, 209-210


def flops_model(t5, lengths, passes=2):
  """Algorithmic FLOPs (2 per multiply-add), SURVEY App. C: (per diffusion step per segment,
  once per segment), with cross K/V hoisted, the unconditional cross-attention elided and the
  FiLM/time tables precomputed."""
  d, hh, F = t5.emb_dim, t5.num_heads * t5.head_dim, t5.mlp_dim
  N, T, C = lengths['targets'], lengths['inputs'], lengths['targets_context']
  M = T + C
  self_attn = 2 * N * d * 3 * hh + 2 * N * hh * d + 2 * 2 * N * N * hh
  cross = 2 * N * d * hh + 2 * N * hh * d + 2 * 2 * N * M * hh
  mlp = 3 * 2 * N * d * F
  inout = 2 * 2 * N * 128 * d
  L = t5.num_decoder_layers
  cond = (self_attn + cross + mlp) * L + inout
  uncond = (self_attn + mlp) * L + inout
  per_step = cond + (uncond if passes == 2 else 0)

  def enc(S):
    return t5.num_encoder_layers * (2 * S * d * 3 * hh + 2 * S * hh * d + 2 * 2 * S * S * hh +
                                    3 * 2 * S * d * F)
  once = L * 2 * M * d * 2 * hh + enc(T) + enc(C)
  return per_step, once


def as_written_flops(t5, lengths):
  """FLOPs of the graph exactly as the reference writes it (what the CPU oracle executes)."""
  d, hh, F = t5.emb_dim, t5.num_heads * t5.head_dim, t5.mlp_dim
  N, T, C = lengths['targets'], lengths['inputs'], lengths['targets_context']
  M = T + C
  L = t5.num_decoder_layers
  self_attn = 2 * N * d * 3 * hh + 2 * N * hh * d + 2 * 2 * N * N * hh
  cross = 2 * N * d * hh + 2 * N * hh * d + 2 * 2 * N * M * hh + 2 * M * d * 2 * hh
  mlp = 3 * 2 * N * d * F
  film = 2 * 2 * 4 * d * 2 * d
  one_pass = (self_attn + cross + mlp + film) * L + 2 * 2 * N * 128 * d + 2 * d * 4 * d + 2 * 16 * d * d
  return 2 * one_pass


def usable_cores() -> int:
  """Host threads this process can really use: affinity mask capped by the cgroup CPU quota."""
  n = len(os.sched_getaffinity(0))
  try:
    with open('/sys/fs/cgroup/cpu.max') as f:
      quota, period = f.read().split()
    if quota != 'max':
      n = max(1, min(n, int(math.ceil(int(quota) / int(period)))))
  except Exception:  # pylint: disable=broad-except
    pass
  return n


def best_thread_count(t5, diff, lengths) -> int:
  """torch-CPU matmuls of this size stop scaling (or regress) with many threads; pick the
  fastest of a few candidates on one decoder layer's worth of work and report it."""
  import torch
  cores = usable_cores()
  cands = sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores}, reverse=True)
  d, F, N = t5.emb_dim, t5.mlp_dim, lengths['inputs'] + lengths['targets_context']
  x = torch.randn(N, d)
  w = torch.randn(d, 2 * F)
  best, best_t = cands[-1], float('inf')
  for c in cands:
    torch.set_num_threads(c)
    for _ in range(2):
      x @ w
    t0 = time.perf_counter()
    for _ in range(6):
      x @ w
    dt = time.perf_counter() - t0
    if dt < best_t * 0.9:
      best, best_t = c, dt
  return best


class ClockSampler(threading.Thread):
  """Samples SM clock / throttle reasons of the local GPU during the timed region."""
  BAD = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20}
  NOTE = {'sw_power_cap': 0x4}

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index = index
    self.samples = []
    self.reasons = set()
    self.max_mhz = None
    self._halt = threading.Event()
    self.ok = False
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
      self.ok = True
    except Exception:  # pylint: disable=broad-except
      self.ok = False

  def run(self):
    if not self.ok:
      return
    while not self._halt.is_set():
      try:
        self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
        mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        for k, bit in {**self.BAD, **self.NOTE}.items():
          if mask & bit:
            self.reasons.add(k)
      except Exception:  # pylint: disable=broad-except
        pass
      self._halt.wait(0.2)

  def finish(self):
    self._halt.set()
    if self.is_alive():
      self.join(timeout=2)
    med = int(np.median(self.samples)) if self.samples else None
    return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
            'samples': len(self.samples)}


def synthetic_batch(B, lengths, seed):
  """SURVEY §8(d): unpadded 2048-token segments, full previous-segment context."""
  rng = np.random.default_rng(seed)
  toks = rng.integers(3, 1391, (B, lengths['inputs'])).astype(np.int32)
  toks[:, -1] = 1
  ctx = rng.uniform(math.log(1e-5), 4.0, (B, lengths['targets_context'], 128)).astype(np.float32)
  cmask = np.ones((B, lengths['targets_context']), np.int32)
  tgt = np.zeros((B, lengths['targets'], 128), np.float32)
  return dict(encoder_input_tokens=toks, encoder_continuous_inputs=ctx,
              encoder_continuous_mask=cmask, decoder_target_tokens=tgt)


def model_configs(args):
  from music_spectrogram_diffusion_b200 import config
  t5 = {'base': config.t5_base, 'small': config.t5_small, 'tiny': config.t5_tiny}[args.model]()
  diff = config.DiffusionConfig()
  diff.sampler.schedule.num_steps = args.diffusion_steps
  # The colab "serve" path runs guidance weight 2.0 (ipynb:223); any weight != 1 costs the same.
  diff.classifier_free_guidance.eval_condition_weight = 2.0
  lengths = dict(config.TASK_FEATURE_LENGTHS_CONTEXT)
  if args.model == 'tiny':
    lengths = {'inputs': 128, 'targets': 128, 'targets_context': 128}
  return t5, diff, lengths


_ORACLE_PARAMS = {}


def cpu_oracle_sample(t5, diff, lengths, n_steps, threads):
  """Time the oracle port (graph AS WRITTEN) on one segment: encode + n_steps full CFG steps;
  returns (seconds_encode, mean seconds per diffusion step, [seconds of every step])."""
  import torch
  from music_spectrogram_diffusion_b200 import weights
  from oracle import msd_oracle as O
  torch.set_num_threads(threads)
  key = (t5.emb_dim, t5.num_decoder_layers, lengths['inputs'])
  if key not in _ORACLE_PARAMS:
    _ORACLE_PARAMS[key] = O.params_to(weights.synthetic_params(
        t5, lengths['inputs'], lengths['targets'], lengths['targets_context'], seed=0))
  params = _ORACLE_PARAMS[key]
  oc = O.OracleConfig(vocab_size=t5.vocab_size, emb_dim=t5.emb_dim, num_heads=t5.num_heads,
                      num_encoder_layers=t5.num_encoder_layers,
                      num_decoder_layers=t5.num_decoder_layers, head_dim=t5.head_dim,
                      mlp_dim=t5.mlp_dim, num_steps=diff.sampler.schedule.num_steps,
                      eval_condition_weight=2.0)
  b = synthetic_batch(1, lengths, seed=0)
  g = torch.Generator().manual_seed(0)
  z = torch.randn(1, lengths['targets'], 128, generator=g)
  with torch.no_grad():
    t0 = time.perf_counter()
    ctx = O.scale_features(torch.from_numpy(b['encoder_continuous_inputs']), oc, clip=True)
    encs = O.encode(params, oc, torch.from_numpy(b['encoder_input_tokens']), ctx,
                    torch.from_numpy(b['encoder_continuous_mask']))
    t_enc = time.perf_counter() - t0

    def pred_fn(zz, time_, cond):
      f = 1.0 if cond else 0.0
      return O.decode(params, oc, [(e * f, m * f) for e, m in encs], zz, time_)

    i0 = oc.num_steps - 1
    per_step = []
    for k in range(n_steps):
      t0 = time.perf_counter()
      z = O.eval_step(z, i0 - k, torch.randn(z.shape, generator=g), pred_fn, oc)
      per_step.append(time.perf_counter() - t0)
  return t_enc, float(np.mean(per_step)), per_step


def cpu_sample_text(cores, n_cpu_steps, t_enc, per_step, num_steps, extra=''):
  """`sample` string of cpu_baseline: says EXTRAPOLATED first, then what was really timed."""
  return (f'EXTRAPOLATED from a bounded sample: oracle port (torch-CPU fp32, graph as written) on '
          f'{cores} threads, 1 segment: encode ({t_enc:.2f} s) + {n_cpu_steps} full CFG diffusion '
          f'steps really timed (mean {np.mean(per_step):.3f} s, min {np.min(per_step):.3f}, max '
          f'{np.max(per_step):.3f}), value = 256 frames / (encode + {num_steps} x mean step); steps '
          f'are identical work and segments independent, so frames/s does not depend on the '
          f'segment count{extra}')


def run_reference(args):
  """--impl reference: the reference's own algorithm on the host cores.  The JAX reference is
  not installable here (no jax/flax/t5x wheels), so this is the oracle port, graph as written.
  Each bench "step" is one bounded sample (encode + --cpu-steps diffusion steps of one segment);
  `ms_per_step` is the measured time of that sample, `value` the frames/s it extrapolates to."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  t5, diff, lengths = model_configs(args)
  cores = best_thread_count(t5, diff, lengths)
  n_cpu_steps = args.cpu_steps
  num_steps = diff.sampler.schedule.num_steps
  secs, samples, all_steps, encs = [], [], [], []
  for it in range(args.warmup + args.steps):
    t0 = time.perf_counter()
    t_enc, t_step, per_step = cpu_oracle_sample(t5, diff, lengths, n_cpu_steps, cores)
    wall = time.perf_counter() - t0
    if it >= args.warmup:
      secs.append(t_enc + num_steps * t_step)
      samples.append(wall)
      all_steps += per_step
      encs.append(t_enc)
  sec = float(np.mean(secs))
  value = lengths['targets'] / sec
  sample = cpu_sample_text(cores, n_cpu_steps, float(np.mean(encs)), all_steps, num_steps,
                           f'; {args.steps} such samples after {args.warmup} warm-up samples')
  line = {
      'impl': 'reference', 'metric': 'mel-frames/sec', 'value': value, 'unit': 'frames/s',
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': float(np.mean(samples)) * 1e3, 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'x_realtime': value / FRAME_RATE, 'extrapolated': True,
      'extrapolated_seconds_per_segment': sec,
      'config': workload_config(args, t5, lengths, segments=args.segments),
      'cpu_baseline': {'value': value, 'unit': 'frames/s', 'cores': cores,
                       'cores_available': usable_cores(), 'kind': 'port', 'sample': sample,
                       'diffusion_steps_timed': len(all_steps),
                       'seconds_per_diffusion_step': {'mean': float(np.mean(all_steps)),
                                                      'min': float(np.min(all_steps)),
                                                      'max': float(np.max(all_steps))}},
      'e2e': {'value': value, 'unit': 'frames/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  print(json.dumps(line))


def workload_config(args, t5, lengths, segments):
  return {
      'workload': f'{args.model}_with_context, {segments} segments/GPU x {lengths["targets"]} '
                  f'frames, {args.diffusion_steps}-step DDPM, CFG weight 2.0, '
                  f'{lengths["inputs"]}-token unpadded MIDI segments + full context',
      'segments_per_gpu': segments, 'diffusion_steps': args.diffusion_steps,
      'emb_dim': t5.emb_dim, 'layers': t5.num_decoder_layers,
      'l2_policy': 'working set per diffusion step (weights 227 MB + cross K/V 85 MB/segment) '
                   'exceeds the 126 MB L2; no explicit flush needed',
      'parallelism': f'dp{args.gpus} (independent segments, no collective in the loop)',
  }


def peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    with open(p) as f:
      j = json.load(f)
    return j.get('bf16_tflops_sustained', 1388.2), j.get('hbm_gbs', 6483.9), 'measured'
  return 1400.0, 6650.0, 'fallback'


KERNEL_CLASS_KEYS = ('gemm', 'attention_combine', 'attention', 'rmsnorm', 'sampler')


def kernel_class(name: str) -> str:
  for k in KERNEL_CLASS_KEYS:
    if k in name:
      return k
  return 'other'


def graph_timeline(eng, seed=2):
  """In-graph timeline of ONE replayed diffusion step (CUPTI through torch.profiler): the per-launch
  CUDA events of `profile_step` serialise the kernels, the replayed graph overlaps every kernel's
  prologue with its predecessor (programmatic dependent launch).  The critical path of a kernel
  is the time it adds to the step: own end - latest end seen before it.  Returns (summary, rows)
  for a step in the middle of an `eng.sample` call, or (None, None) if CUPTI is unavailable."""
  import tempfile
  import torch
  try:
    for _ in range(2):
      eng.sample(seed=1)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
      eng.sample(seed=seed)
      torch.cuda.synchronize()
    path = os.path.join(tempfile.mkdtemp(), 'trace.json')
    prof.export_chrome_trace(path)
    with open(path) as f:
      ev = [e for e in json.load(f)['traceEvents'] if e.get('cat') == 'kernel']
  except Exception as e:  # pylint: disable=broad-except
    return {'unavailable': f'{type(e).__name__}: {e}'}, None
  ev.sort(key=lambda e: e['ts'])
  # the call = a few set-up kernels (noise draw) + num_steps identical graph replays
  steps = int(eng.cfg.num_steps)
  pre = next((k for k in range(4) if (len(ev) - k) % steps == 0 and len(ev) > k), None)
  if pre is None or steps < 4:
    return {'unavailable': f'{len(ev)} kernels do not split into {steps} equal steps'}, None
  nodes = (len(ev) - pre) // steps
  lo = pre + (steps // 2) * nodes
  step = ev[lo:lo + nodes]
  t0 = step[0]['ts']
  rows, crit, busy = [], {}, {}
  prev_end = t0
  for e in step:
    c = kernel_class(e['name'])
    end = e['ts'] + e['dur']
    add = max(0.0, end - prev_end)
    rows.append({'kernel': c, 'start_us': round(e['ts'] - t0, 2), 'dur_us': round(e['dur'], 2),
                 'critical_us': round(add, 2), 'grid': e.get('args', {}).get('grid'),
                 'block': e.get('args', {}).get('block')})
    crit[c] = crit.get(c, 0.0) + add
    busy[c] = busy.get(c, 0.0) + e['dur']
    prev_end = max(prev_end, end)
  total = prev_end - t0
  summary = {'kernels': len(step), 'step_us': round(total, 1),
             'critical_path_us_by_class': {k: round(v, 1) for k, v in crit.items()},
             'critical_path_share_by_class': {k: round(v / total, 4) for k, v in crit.items()},
             'busy_us_by_class': {k: round(v, 1) for k, v in busy.items()},
             'how': 'CUPTI kernel records of one replayed step graph; critical = own end - latest '
                    'earlier end'}
  return summary, rows


def measure_gemm_traffic(args, timeout_s=240):
  """dram__bytes_read + write of the dominant kernel (CTA-pair GEMM), per launch, from an ncu pass
  over one uncaptured diffusion step of this very workload (tools/profile_step.py in a child
  process; two metrics = one replay pass).  Returns a dict, or {'unavailable': why}."""
  import shutil
  import subprocess
  import tempfile
  ncu = shutil.which('ncu') or ('/usr/local/cuda/bin/ncu' if os.path.exists('/usr/local/cuda/bin/ncu') else None)
  if ncu is None:
    return {'unavailable': 'ncu not found'}
  log = os.path.join(tempfile.mkdtemp(), 'traffic.csv')
  # encode issues 109 GEMM launches for base (2 encoders x 12 layers x 4 + context input
  # projection + 12 cross K/V), then one warm-up step of 74 and the measured one
  skip = {'base': 109 + 74}.get(args.model)
  if skip is None or args.precision != 'bf16':
    return {'unavailable': 'launch indices are tabulated for the base bf16 workload only'}
  cmd = [ncu, '--metrics', 'dram__bytes_read.sum,dram__bytes_write.sum', '--clock-control', 'none',
         '-k', 'regex:gemm_bf16_tcgen05_pair', '-s', str(skip), '-c', '74', '--csv', '--log-file', log,
         sys.executable, os.path.join(ROOT, 'tools', 'profile_step.py'), '--model', args.model,
         '--segments', str(args.segments), '--diffusion-steps', str(args.diffusion_steps)]
  try:
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s)
  except Exception as e:  # pylint: disable=broad-except
    return {'unavailable': f'{type(e).__name__}: {e}'}
  if not os.path.exists(log):
    return {'unavailable': f'ncu wrote no log (rc {r.returncode}): {r.stderr[-200:]}'}
  import csv
  total, ids = 0.0, set()
  with open(log) as f:
    lines = [ln for ln in f if not ln.startswith('==')]
  for row in csv.DictReader(lines):
    name = row.get('Metric Name', '')
    if name.startswith('dram__bytes_'):
      try:
        v = float(row['Metric Value'].replace(',', ''))
      except ValueError:
        continue
      unit = row.get('Metric Unit', 'byte').lower()
      v *= {'byte': 1.0, 'kbyte': 1e3, 'mbyte': 1e6, 'gbyte': 1e9}.get(unit, 1.0)
      total += v
      ids.add(row.get('ID'))
  if not ids:
    return {'unavailable': f'no dram__bytes rows in the ncu log (rc {r.returncode}): '
                           f'{(r.stderr or r.stdout)[-200:]}'}
  return {'dram_bytes_per_launch': total / len(ids), 'launches': len(ids),
          'how': 'ncu dram__bytes_read.sum + dram__bytes_write.sum over the 74 CTA-pair GEMM '
                 'launches of one uncaptured diffusion step, measured in this run'}


DUMP_BUDGET_BYTES = 60_000_000  # under 64 MB (decimal or binary) with the .npy headers and index file


def dump_outputs(directory, name, mel, budget=DUMP_BUDGET_BYTES):
  """Writes `mel` [segments, frames, n_dims] as <directory>/<name>.npy (float32), so that two
  builds can be compared output for output.  Past `budget` bytes it writes a fixed seeded sample
  of whole segments instead, and their indices as <name>_segments.npy."""
  mel = mel.float().cpu().numpy()
  os.makedirs(directory, exist_ok=True)
  keep = budget // (mel[0].nbytes + 8)
  if mel.shape[0] > keep:
    idx = np.sort(np.random.default_rng(0).choice(mel.shape[0], keep, replace=False))
    mel = mel[idx]
    np.save(os.path.join(directory, f'{name}_segments.npy'), idx.astype(np.float64))
  np.save(os.path.join(directory, f'{name}.npy'), mel)


def synthetic_song_notes(segments, lengths):
  """A multi-instrument synthetic arrangement covering `segments` 5.12 s segments."""
  from music_spectrogram_diffusion_b200 import midi_tokens
  rng = np.random.default_rng(5)
  seconds = segments * lengths['targets'] / FRAME_RATE - 0.25
  rows = []
  for program in (0, 25, 33, 48, 56):
    t = float(rng.uniform(0, 0.3))
    while t < seconds - 0.3:
      d = float(rng.uniform(0.1, 0.9))
      rows.append((t, min(t + d, seconds), int(rng.integers(36, 84)), int(rng.integers(30, 127)),
                   program, False))
      t += float(rng.uniform(0.08, 0.4))
  return midi_tokens.make_notes(rows), len(rows)


def single_song_sample(t5, diff, lengths, device_index, segments=12, world=1):
  """BASELINE config 5: ONE synthetic multi-instrument song of `segments` chained 5.12 s segments
  (61.44 s for 12; batch 1, context = previous prediction), timed like the reference's
  `model_timing` (first segment excluded, beam/evaluation.py:217-220).
  N = 1: song.synthesize_song through InferenceModel.predict (host batches, as the reference).
  N >= 2: ranks 0 and 1 split the classifier-free guidance (conditional pass on one GPU,
  unconditional on the other, predicted noise exchanged by NVLink stores inside the sampler
  kernel: distributed.synthesize_song_cfg_split); the chain is serial, so further ranks cannot
  help this one song and only join the barriers."""
  import torch
  from music_spectrogram_diffusion_b200 import distributed as D, inference, midi_tokens, song
  notes, n_notes = synthetic_song_notes(segments, lengths)
  model = inference.InferenceModel.from_config(t5, diff, lengths, 'synthetic:0', 1, device_index)
  ac = model.audio_codec
  seconds_per_chunk = lengths['targets'] * (ac.hop_size / ac.sample_rate)
  if world == 1:
    out = song.synthesize_song(model, notes, seed=0)
    timing = out['model_timing']
    per_chunk = timing['prediction_seconds_per_chunk']
    toks = out['tokens']
    api = 'song.synthesize_song(InferenceModel(batch_size=1), notes): tokenise + chained predict'
    gpus_used = 1
  else:
    import torch.distributed as dist
    tk = midi_tokens.tokenize_song(
        notes, song.event_vocabulary_of(model), inputs_length=lengths['inputs'],
        frames_per_segment=lengths['targets'], frame_rate=ac.frame_rate, sample_rate=ac.sample_rate,
        hop_size=ac.hop_size)
    toks = tk.tokens
    segs = [torch.from_numpy(np.ascontiguousarray(t)) for t in toks]
    model.engine  # build before the handles are swapped
    timings = []
    mel = D.synthesize_song_cfg_split(model, segs, lengths['targets_context'], 128, seed=0,
                                      timings=timings)
    dist.barrier()
    if mel is None or dist.get_rank() != 0:
      del model
      return None
    per_chunk = float(np.mean(timings))
    api = ('distributed.synthesize_song_cfg_split: conditional pass on GPU 0, unconditional on GPU 1, '
           'eps exchanged by peer stores inside the sampler kernel; device-resident chain')
    gpus_used = 2
  del model
  return {
      'segments': int(len(toks)), 'notes': n_notes, 'audio_seconds': len(toks) * seconds_per_chunk,
      'tokens_per_segment': [int((r > 0).sum()) for r in toks],
      'seconds_per_segment': per_chunk,
      'x_realtime': seconds_per_chunk / per_chunk,
      'gpus_used_by_this_song': gpus_used,
      'api': api,
  }


def run_ours(args):
  import torch
  import torch.distributed as dist
  from music_spectrogram_diffusion_b200 import engine as eng_mod
  from music_spectrogram_diffusion_b200 import inference

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  dev = torch.device('cuda', local)
  torch.cuda.set_device(dev)

  t5, diff, lengths = model_configs(args)
  B = args.segments
  model = inference.InferenceModel.from_config(
      t5, diff, lengths, checkpoint_path='synthetic:0', batch_size=B, device=local,
      precision=args.precision)
  eng = model.engine
  batch = synthetic_batch(B, lengths, seed=100 + rank)
  d_tok = torch.from_numpy(batch['encoder_input_tokens']).to(dev)
  d_ctx = torch.from_numpy(batch['encoder_continuous_inputs']).to(dev)
  d_msk = torch.from_numpy(batch['encoder_continuous_mask']).to(dev)
  d_mel = torch.empty(B, lengths['targets'], 128, device=dev)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize(dev)

  def device_step():
    eng.encode(d_tok, d_ctx, d_msk)
    eng.sample(None, None, seed=0, out=d_mel)

  def host_step():
    return model.predict(batch, seed=0)

  def timed(fn, warmup, steps):
    for _ in range(warmup):
      fn()
    barrier()
    launches0 = eng_mod.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
      fn()
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.finish()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / 1e3, wall, clocks, eng_mod.launch_count() - launches0

  sec, wall, clocks, launches = timed(device_step, args.warmup, args.steps)
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, 'mel' if world == 1 else f'mel_rank{rank}', d_mel,
                 DUMP_BUDGET_BYTES // world)
  frames = world * B * lengths['targets'] * args.steps
  value = frames / sec
  sec_e2e, wall_e2e, clocks_e2e, _ = timed(host_step, max(1, args.warmup // 2), args.steps)
  value_e2e = frames / sec_e2e

  # ---- BASELINE config 5: one chained song (every rank takes part in the set-up barriers) ----
  song_result = None
  if not args.no_song and lengths['inputs'] >= 2048 and args.precision == 'bf16':
    song_result = single_song_sample(t5, diff, lengths, local, segments=args.song_segments,
                                     world=world)

  # ---- roofline of the dominant kernel class (tcgen05 GEMM), CUDA events per launch -------
  prof = None
  if rank == 0:
    eng.encode(d_tok, d_ctx, d_msk)
    prof = eng.profile_step(step_i=args.diffusion_steps // 2 or 1, reps=3)
    torch.cuda.synchronize(dev)
  peak_tf, peak_hbm, peak_kind = peaks()
  per_step, once = flops_model(t5, lengths)
  alg_flops_per_frame = (per_step * args.diffusion_steps + once) / lengths['targets']

  if rank == 0:
    total_ms = sum(v['ms'] for v in prof.values())
    g = prof['gemm']
    gemm_tf = g['flops'] / (g['ms'] * 1e-3) / 1e12 if g['ms'] > 0 else 0.0
    a = prof['attention']
    attn_tf = a['flops'] / (a['ms'] * 1e-3) / 1e12 if a['ms'] > 0 else 0.0
    # in-graph critical path (what the replayed graph really spends per kernel class)
    timeline = None
    if not args.no_timeline:
      eng.encode(d_tok, d_ctx, d_msk)
      timeline, _ = graph_timeline(eng)
    # DRAM traffic of the dominant kernel, measured in this run when ncu may read the counters
    traffic, traffic_info = None, {'unavailable': 'skipped (--no-traffic or N > 1)'}
    if world == 1 and not args.no_traffic:
      traffic_info = measure_gemm_traffic(args)
      traffic = traffic_info.get('dram_bytes_per_launch')
    if traffic is None:
      tpath = os.path.join(ROOT, 'profiles', 'gemm_traffic.json')
      if os.path.exists(tpath):
        with open(tpath) as f:
          traffic = json.load(f).get('dram_bytes_per_launch')
        traffic_info = dict(traffic_info, fallback='profiles/gemm_traffic.json (recorded by an '
                            'earlier ncu --set full capture, not measured in this run)')
    g_crit = (timeline or {}).get('critical_path_us_by_class', {}).get('gemm')
    roofline = {
        'kernel': 'gemm_bf16_tcgen05_pair_kernel', 'bound': 'tensor',
        'achieved': gemm_tf, 'peak': peak_tf, 'unit': 'TFLOP/s',
        'frac': gemm_tf / peak_tf, 'peak_source': f'{peak_kind} (bf16 sustained)',
        'traffic': traffic, 'traffic_source': traffic_info,
        'algorithmic_bytes_per_launch': g['bytes'] / max(g['launches'], 1),
        # the same FLOPs over the time the class adds to the replayed step graph (PDL overlap)
        'achieved_in_graph': (g['flops'] / (g_crit * 1e-6) / 1e12) if g_crit else None,
        'frac_in_graph': (g['flops'] / (g_crit * 1e-6) / 1e12 / peak_tf) if g_crit else None,
        'launches_per_diffusion_step': g['launches'],
        'avg_launch_us': 1e3 * g['ms'] / max(g['launches'], 1),
        'share_of_step': g['ms'] / total_ms if total_ms > 0 else None,
        'how': 'CUDA events around every launch of one uncaptured diffusion step (3 reps)',
        # bf16 mode: the decoder layers' 36 pre-norms (+FiLM) run inside these launches' epilogues
        # (deferred normalisation, DESIGN section 3), so their time is GEMM time here while the
        # FLOP count is the projections' alone; MSD_FUSED_NORM=0 gives the round-1 accounting
        'includes': 'pre-norm + FiLM of the decoder layers (no stand-alone rmsnorm kernels)'
                    if os.environ.get('MSD_FUSED_NORM', '1') != '0' and args.precision == 'bf16' else None,
    }
    step_tf = alg_flops_per_frame * (value / world) / 1e12
    line = {
        'metric': 'mel-frames/sec', 'value': value, 'unit': 'frames/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'bf16' if args.precision == 'bf16' else
                 'f32 (3 x bf16 split tensor-core products ~2^-16, fp32 attention / softmax / residual)',
        'data': 'synthetic',
        'x_realtime': value / FRAME_RATE,
        'config': workload_config(args, t5, lengths, B),
        'clocks': clocks,
        'e2e': {'value': value_e2e, 'unit': 'frames/s',
                'h2d_bytes_per_step': int(sum(batch[k].nbytes for k in (
                    'encoder_input_tokens', 'encoder_continuous_inputs',
                    'encoder_continuous_mask'))),
                'd2h_bytes_per_step': int(B * lengths['targets'] * 128 * 4),
                'x_realtime': value_e2e / FRAME_RATE, 'clocks': clocks_e2e,
                'api': 'InferenceModel.predict(host numpy batch) incl. pinned H2D and D2H'},
        'gpu_launches': int(launches),
        'roofline': roofline,
        'whole_step': {
            'algorithmic_gflop_per_frame': alg_flops_per_frame / 1e9,
            'achieved_tflops_per_gpu': step_tf, 'frac_of_peak': step_tf / peak_tf,
            'wall_seconds': wall,
        },
        'kernel_classes_ms_per_diffusion_step': {k: round(v['ms'], 4) for k, v in prof.items()},
        'in_graph': timeline,
        'attention_tflops': attn_tf,
    }
    if song_result is not None:
      line['single_song'] = song_result
    if world == 1 and not args.no_cpu_baseline:
      cores = best_thread_count(t5, diff, lengths)
      t_enc, t_step, per_step = cpu_oracle_sample(t5, diff, lengths, args.cpu_steps, cores)
      cpu_sec = t_enc + args.diffusion_steps * t_step
      line['cpu_baseline'] = {
          'value': lengths['targets'] / cpu_sec, 'unit': 'frames/s', 'cores': cores,
          'cores_available': usable_cores(), 'kind': 'port', 'extrapolated': True,
          'sample': cpu_sample_text(cores, args.cpu_steps, t_enc, per_step, args.diffusion_steps,
                                    f' ({as_written_flops(t5, lengths) / 1e9:.1f} GFLOP per step)'),
          'seconds_per_diffusion_step': {'mean': float(np.mean(per_step)),
                                         'min': float(np.min(per_step)),
                                         'max': float(np.max(per_step))},
      }
    print(json.dumps(line))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=3)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--model', default='base', choices=['base', 'small', 'tiny'])
  ap.add_argument('--segments', type=int, default=8, help='segments per GPU (B)')
  ap.add_argument('--diffusion-steps', type=int, default=1000)
  ap.add_argument('--cpu-steps', type=int, default=10,
                  help='diffusion steps in the bounded CPU sample')
  ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32_accurate'],
                  help='fp32_accurate: BASELINE config 2 (use with --segments 1)')
  ap.add_argument('--no-timeline', action='store_true',
                  help='skip the in-graph (CUPTI) critical-path split per kernel class')
  ap.add_argument('--no-traffic', action='store_true',
                  help='skip the ncu DRAM-traffic measurement of the dominant kernel')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-song', action='store_true',
                  help='skip the batch-1 chained-song sample (BASELINE config 5)')
  ap.add_argument('--song-segments', type=int, default=12,
                  help='segments of the chained song (12 = 61.44 s, BASELINE config 5)')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='after the timed steps, write the mel batch of the last one as DIR/mel.npy '
                       '(DIR/mel_rank<r>.npy per rank under torchrun)')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs writes the outputs of --impl ours')
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
