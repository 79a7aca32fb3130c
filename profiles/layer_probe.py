"""Per-layer GEMM timing of the Mnih'15 Q-network at batch 256 (config 2 shapes): forward, input
gradient (dX) and parameter gradient (dW + db) of every layer, each timed as R back-to-back
launches replayed from one CUDA graph (CUDA events on the launch stream; the number is kernel
time, not Python launch overhead).

    python profiles/layer_probe.py [--reps 20] [--batch 256]

Prints one JSON line per (layer, pass).  `gflop` is the fp32-equivalent work of the GEMM,
`tflops` = gflop / time.  Used by profiles/README.md's per-layer table.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from agents_b200 import _lib  # noqa: E402
from agents_b200.networks import layers as L  # noqa: E402
from agents_b200.networks import q_network  # noqa: E402
from agents_b200.specs import tensor_spec  # noqa: E402

def timed_graph(fn, reps, iters=5):
  """Captures `reps` calls of fn into one graph, replays it `iters` times; returns us per call."""
  for _ in range(2):
    fn()
  torch.cuda.synchronize()
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g):
    for _ in range(reps):
      fn()
  g.replay()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  best = None
  for _ in range(iters):
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e3 / reps
    best = t if best is None else min(best, t)
  return best


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--reps', type=int, default=20)
  ap.add_argument('--batch', type=int, default=256)
  args = ap.parse_args()
  dev = torch.device('cuda:0')
  obs_spec = tensor_spec.TensorSpec((84, 84, 4), torch.uint8)
  act_spec = tensor_spec.BoundedTensorSpec((), torch.int32, 0, 5)
  net = q_network.QNetwork(obs_spec, act_spec, preprocessing_layers=L.CastScale(255.),
                           conv_layer_params=((32, 8, 4), (64, 4, 2), (64, 3, 1)),
                           fc_layer_params=(512,), device=dev).set_seed(0)
  net.create_variables()
  B = args.batch
  x = torch.randint(0, 256, (B, 84, 84, 4), dtype=torch.uint8, device=dev)
  layers = [l for l in net.layers if not isinstance(l, L.CastScale)]
  acts, h = [], x
  for l in layers:
    y = l.forward(h)
    acts.append((l, h, y))
    h = y
  torch.cuda.synchronize()
  names = iter(['conv1', 'conv2', 'conv3', 'flatten', 'fc1', 'fc2'])
  prev_act = 0
  for i, (l, xin, y) in enumerate(acts):
    name = next(names)
    if not hasattr(l, 'backward_parts'):
      continue
    dz = torch.randn_like(y)
    if isinstance(l, L.Conv2D):
      m, n, k = B * l.oh * l.ow, l.filters, l.kh * l.kw * l.c
    else:
      m, n, k = B, l.units, l.in_features
    gflop = 2.0 * m * n * k / 1e9
    passes = [('fwd', lambda l=l, xin=xin: l.forward(xin))]
    if xin.dtype != torch.uint8:
      passes.append(('dX', lambda l=l, xin=xin, dz=dz: l.backward_parts(xin, dz, True, False,
                                                                         x_act=prev_act)))
      passes.append(('dX_nomask', lambda l=l, xin=xin, dz=dz: l.backward_parts(xin, dz, True, False)))
    passes.append(('dW', lambda l=l, xin=xin, dz=dz: l.backward_parts(xin, dz, False, True,
                                                                      accumulate=1)))
    for pname, fn in passes:
      us = timed_graph(fn, args.reps)
      line = dict(layer=name, op=pname, M=m, N=n, K=k, us=round(us, 2), gflop=round(gflop, 3),
                  tflops=round(gflop / us * 1e-3 * 1e6 / 1e3, 2))
      print(json.dumps(line), flush=True)
    prev_act = l._act
  # separate kernels that the fused paths replace / that remain on the step
  y1 = acts[0][2]
  dy1 = torch.randn_like(y1)
  us = timed_graph(lambda: acts[0][0].backward_act(y1, dy1), args.reps)
  print(json.dumps(dict(layer='conv1', op='act_bwd(separate kernel)', us=round(us, 2))), flush=True)
  # whole net forward / backward as the agent runs them (eager launch order, one graph)
  dq = torch.randn(B, 6, device=dev)

  def fwd():
    return net.forward_train(x)

  q, tape = fwd()
  us_f = timed_graph(fwd, 5)
  us_b = timed_graph(lambda: net.backward(tape, dq), 5)
  print(json.dumps(dict(layer='net', op='forward_train', us=round(us_f, 1))), flush=True)
  print(json.dumps(dict(layer='net', op='backward(graph: dW side stream)', us=round(us_b, 1))),
        flush=True)


if __name__ == '__main__':
  main()
