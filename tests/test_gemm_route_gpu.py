"""Which GEMM engine each dense / conv shape runs on: the kernel names of one eager call, read with
torch.profiler.  Modes 1 and 2 send a GEMM to the tensor-core kernel (tc2_gemm_kernel) when
N >= 16, M >= 32, K >= 8 and both operands can be read as aligned 16-byte chunks, and to the fp32
FFMA kernel (sgemm_kernel) otherwise; inputs of <= 32 features and heads of <= 16 outputs have
kernels of their own (thin_*, skinny_*).  These tests pin the route of the benchmarked networks'
layers, so that a dispatch change cannot silently move them to a slower engine."""
import os

import numpy as np
import pytest
import torch

from agents_b200 import _lib
from agents_b200.networks import layers as L
from oracle import nn as onn
from conftest import record_parity

pytestmark = pytest.mark.gpu
f32 = np.float32
TC2, FFMA = 'tc2_gemm_kernel', 'sgemm_kernel'


def _kernels(fn):
  """Names of the kernels one call of fn launches (after a warm-up call outside the trace)."""
  fn()
  torch.cuda.synchronize()
  with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    fn()
    torch.cuda.synchronize()
  names = [e.key for e in prof.key_averages()]
  assert any('b200rl' in n for n in names), f'no kernel of the library in the trace: {names}'
  return names


def _assert_route(fn, want, where):
  names = _kernels(fn)
  assert any(want in n for n in names), (where, want, names)
  if want != FFMA:
    assert not any(FFMA in n for n in names), (where, names)
  if want != TC2:
    assert not any(TC2 in n for n in names), (where, names)


def _bind(layer, in_shape, gen, pre_divisor=None):
  layer.build(in_shape)
  ps = [torch.randn(*s, device='cuda', generator=gen) * 0.05 for s in layer.param_shapes()]
  layer.bind(ps, [torch.zeros_like(p) for p in ps])
  if pre_divisor is not None:
    layer.pre_divisor = pre_divisor
  return layer


def _passes(layer, x, need_dx):
  """fwd / dX / dW calls of one layer as the networks make them."""
  y = layer.forward(x)
  dz = torch.randn_like(y)
  out = {'fwd': lambda: layer.forward(x),
         'dW': lambda: layer.backward_parts(x, dz, False, True, accumulate=1)}
  if need_dx:
    out['dX'] = lambda: layer.backward_parts(x, dz, True, False)
  return y, out


def _check_stack(cuda, x, layers, pre_divisor=None):
  """layers: (name, layer, {pass: expected kernel}); the output of each layer feeds the next."""
  gen = torch.Generator(device=cuda).manual_seed(0)
  h = x
  for i, (name, layer, want) in enumerate(layers):
    if isinstance(layer, L.Dense) and h.dim() > 2:
      h = h.reshape(h.shape[0], -1)
    _bind(layer, tuple(h.shape[1:]), gen, pre_divisor if i == 0 else None)
    y, passes = _passes(layer, h, need_dx='dX' in want)
    assert set(passes) == set(want), (name, sorted(passes))
    for p, kernel in want.items():
      _assert_route(passes[p], kernel, f'{name}.{p}')
    h = y


def _mode_default():
  return int(os.environ.get('B200RL_GEMM_MODE', '1'))


def test_mnih15_net_at_batch_256_runs_on_tc2(cuda):
  x = torch.randint(0, 256, (256, 84, 84, 4), dtype=torch.uint8, device=cuda)
  all3 = {'fwd': TC2, 'dX': TC2, 'dW': TC2}
  _check_stack(cuda, x, [
      ('conv1', L.Conv2D(32, 8, 4, activation='relu'), {'fwd': TC2, 'dW': TC2}),
      ('conv2', L.Conv2D(64, 4, 2, activation='relu'), all3),
      ('conv3', L.Conv2D(64, 3, 1, activation='relu'), all3),
      ('fc1', L.Dense(512, activation='relu'), all3)], pre_divisor=255.0)


@pytest.mark.parametrize('name,rows,obs,hidden,head', [
    ('ppo_actor', 4096, 17, (200, 100), 6), ('ppo_value', 4096, 17, (200, 100), 1),
    ('sac_actor', 256, 17, (256, 256), 12), ('sac_critic', 256, 23, (256, 256), 1)])
def test_mlp_layers_take_thin_tc2_and_skinny_kernels(cuda, name, rows, obs, hidden, head):
  act = 'tanh' if name.startswith('ppo') else 'relu'
  x = torch.randn(rows, obs, device=cuda)
  _check_stack(cuda, x, [
      (f'{name}.in', L.Dense(hidden[0], activation=act), {'fwd': 'thin_fwd', 'dW': 'thin_dw'}),
      (f'{name}.hidden', L.Dense(hidden[1], activation=act), {'fwd': TC2, 'dX': TC2, 'dW': TC2}),
      (f'{name}.head', L.Dense(head), {'fwd': 'skinny_fwd', 'dX': 'skinny_dx', 'dW': 'skinny_dw'})])


def test_shapes_tc2_cannot_vectorise_take_ffma(cuda):
  """K = 65 and N = 129 are not multiples of 4; a uint8 input with C = 1 cannot be copied in
  16-byte chunks of whole patch rows.  Both run on the FFMA kernel in mode 1."""
  gen = torch.Generator(device=cuda).manual_seed(1)
  dense = _bind(L.Dense(129, activation='relu'), (65,), gen)
  _, passes = _passes(dense, torch.randn(33, 65, device=cuda), need_dx=True)
  for p, fn in passes.items():
    _assert_route(fn, FFMA, f'dense_33x65x129.{p}')
  conv = _bind(L.Conv2D(16, 3, 1, activation='relu'), (10, 10, 1), gen, pre_divisor=255.0)
  x = torch.randint(0, 256, (5, 10, 10, 1), dtype=torch.uint8, device=cuda)
  _, passes = _passes(conv, x, need_dx=False)
  for p, fn in passes.items():
    _assert_route(fn, FFMA, f'conv_u8_c1.{p}')


def test_mode2_atari_conv1_raw_pixels_on_tc2(cuda):
  """Mode 2 (1xTF32) takes the uint8 conv1 on tc2 with the raw-pixel view: A is exact in TF32,
  so only the weights / dY are rounded (~1e-3 of the largest element is documented for 1xTF32)."""
  rng = np.random.RandomState(7)
  x = rng.randint(0, 256, size=(32, 84, 84, 4)).astype(np.uint8)
  xt = torch.as_tensor(x, device=cuda)
  conv = _bind(L.Conv2D(32, 8, 4, activation='relu'), (84, 84, 4),
               torch.Generator(device=cuda).manual_seed(2), pre_divisor=255.0)
  with torch.no_grad():
    conv.bias.copy_(torch.as_tensor(rng.randn(32).astype(f32) * 0.1))
  dz = rng.randn(32, conv.oh, conv.ow, 32).astype(f32)
  dzt = torch.as_tensor(dz, device=cuda)
  w, b = conv.kernel.cpu().numpy(), conv.bias.cpu().numpy()
  xf = (x.astype(f32) / f32(255.0)).astype(f32)
  want_y = onn.conv2d_fwd(xf, w, b, 4, 'relu')
  _, want_dw, want_db = onn.conv2d_bwd(xf, w, dz, 4, need_dx=False)
  _lib.call('b200rl_set_gemm_mode', 2)
  try:
    _assert_route(lambda: conv.forward(xt), TC2, 'conv1.fwd')
    _assert_route(lambda: conv.backward_parts(xt, dzt, False, True), TC2, 'conv1.dW')
    y = conv.forward(xt).cpu().numpy()
    conv.backward_parts(xt, dzt, False, True)
    got = dict(fwd=(y, want_y), dW=(conv.d_kernel.cpu().numpy(), want_dw),
               db=(conv.d_bias.cpu().numpy(), want_db))
  finally:
    _lib.call('b200rl_set_gemm_mode', _mode_default())
  errs = {k: float(np.abs(g - v).max() / np.abs(v).max()) for k, (g, v) in got.items()}
  record_parity('mode2_atari_conv1_err_rel_to_max', **errs)
  for k, e in errs.items():
    assert e <= 2e-3, (k, errs)


def test_dqn_parity_net_runs_every_layer_on_tc2(cuda):
  """The net of test_baseline_parity_gpu.py::test_dqn_train_parity_all_layers_on_tensor_cores."""
  x = torch.randint(0, 256, (32, 28, 28, 4), dtype=torch.uint8, device=cuda)
  all3 = {'fwd': TC2, 'dX': TC2, 'dW': TC2}
  _check_stack(cuda, x, [
      ('conv1', L.Conv2D(16, 4, 4, activation='relu'), {'fwd': TC2, 'dW': TC2}),
      ('conv2', L.Conv2D(32, 3, 1, activation='relu'), all3),
      ('fc1', L.Dense(64, activation='relu'), all3)], pre_divisor=255.0)
