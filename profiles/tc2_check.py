"""tc2 (persistent cp.async tcgen05 GEMM) against the fp32 FFMA engine (gemm mode 0), layer by layer:
max relative difference and time of forward / dX / dW for the Mnih'15 layers (batch 256), the
PPO (200,100) tanh MLP at 4096x128 rows and the SAC (256,256) critic at batch 1024.
A progress line is flushed BEFORE every launch, so a hang names its culprit.

    python profiles/tc2_check.py [--reps 20] [--flags 0]   # --flags 1: explicitly masked hi plane; 4: no TMA
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from agents_b200 import _lib  # noqa: E402
from agents_b200.networks import layers as L  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument('--reps', type=int, default=20)
ap.add_argument('--flags', type=int, default=0)
ap.add_argument('--only', default='')
args = ap.parse_args()
dev = torch.device('cuda:0')
_lib.call('b200rl_set_tc2_flags', args.flags)
gen = torch.Generator(device=dev).manual_seed(0)


def bind(layer, in_shape):
  layer.build(in_shape)
  ps = [torch.randn(*s, device=dev, generator=gen) * 0.05 for s in layer.param_shapes()]
  gs = [torch.zeros_like(p) for p in ps]
  layer.bind(ps, gs)
  return layer, gs


def timed(fn, reps):
  fn()
  torch.cuda.synchronize()
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g):
    for _ in range(reps):
      fn()
  g.replay()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  best = 1e9
  for _ in range(3):
    e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1) * 1e3 / reps)
  return best


def rel(a, b):
  return float((a - b).abs().max() / b.abs().max().clamp_min(1e-20))


def say(**kw):
  print(json.dumps(kw), flush=True)


def run_both(name, op, fn, outs):
  """fn() runs the op and returns the tensors to compare."""
  if args.only and args.only not in f'{name}.{op}':
    return
  res = {}
  for tag, mode in (('ffma', 0), ('tc2', 1)):
    say(progress=f'{name}.{op}.{tag}')
    _lib.call('b200rl_set_gemm_mode', mode)
    o = fn()
    torch.cuda.synchronize()
    res[tag] = [t.clone() for t in o]
    res[tag + '_us'] = timed(fn, args.reps)
  diffs = [rel(x, y) for x, y in zip(res['tc2'], res['ffma'])]
  say(layer=name, op=op, ffma_us=round(res['ffma_us'], 2), tc2_us=round(res['tc2_us'], 2),
      speedup=round(res['ffma_us'] / res['tc2_us'], 2), max_rel_diff=max(diffs), outs=outs)


def check_layer(name, layer, x, prev_act):
  layer, gs = bind(layer, tuple(x.shape[1:]))
  y = layer.forward(x)
  dz = torch.randn(y.shape, device=dev, generator=gen)
  run_both(name, 'fwd', lambda: [layer.forward(x)], ['y'])
  if x.dtype != torch.uint8:
    run_both(name, 'dX', lambda: [layer.backward_parts(x, dz, True, False, x_act=prev_act)], ['dx'])

  def dw():
    for g in gs:
      g.zero_()
    layer.backward_parts(x, dz, False, True, accumulate=1)
    return gs
  run_both(name, 'dW', dw, ['dkernel', 'dbias'])
  return y


B = 256
x = torch.randint(0, 256, (B, 84, 84, 4), dtype=torch.uint8, device=dev, generator=gen)
c1 = L.Conv2D(32, 8, 4, activation='relu'); c1.pre_divisor = 255.0
h = check_layer('conv1', c1, x, 0)
h = check_layer('conv2', L.Conv2D(64, 4, 2, activation='relu'), h, 1)
h = check_layer('conv3', L.Conv2D(64, 3, 1, activation='relu'), h, 1)
h = h.reshape(B, -1)
h = check_layer('fc1', L.Dense(512, activation='relu'), h, 1)
# odd sizes: ragged M / N tiles, K not a multiple of 32
xr = torch.randn(1000, 200, device=dev, generator=gen)
check_layer('ragged_1000x200x100', L.Dense(100, activation='tanh'), xr, 2)
# PPO MLP (4096 x 128 rows; the 17-wide input layer has kernels of its own)
xp = torch.randn(4096 * 128, 200, device=dev, generator=gen).tanh()
check_layer('ppo_200x100', L.Dense(100, activation='tanh'), xp, 2)
# SAC critic
xs = torch.randn(1024, 256, device=dev, generator=gen).relu()
check_layer('sac_256x256', L.Dense(256, activation='relu'), xs, 1)
_lib.call('b200rl_set_tc2_flags', 0)
_lib.call('b200rl_set_gemm_mode', 1)
say(done=True)
