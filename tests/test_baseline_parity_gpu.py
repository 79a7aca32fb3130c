"""Full train-step parity AT the BASELINE.json configurations (VERDICT r1, "Next round" item 1).

The layer- and kernel-level tests run small shapes; these run >= 3 complete train steps at the
benchmark shapes and compare loss / per-example td_error / post-step parameters with the oracle:

  config 2  Mnih'15 Q-net, batch 256, T=2, centered RMSProp, tcgen05 3xTF32 path end to end
            (oracle/dqn_torch.py, cross-checked against oracle/dqn.py in tests/test_oracle_nn.py)
  config 3  PPO (200, 100) tanh nets, T=128, both normalisers ON, 2 epochs x 2 train calls; the
            4096 trajectories are cut to 512 so that the numpy oracle stays within seconds
  config 4  SAC (256, 256) relu nets, batch 1024, 3 steps
  conv net with 16 / 32 filters, batch 32: every conv/dense GEMM of a 5-step DQN run on the
            tensor-core path (the small nets of tests/test_dqn_gpu.py keep conv1 on FFMA).

Tolerances: losses 1e-5 relative (north_star).  Quantities that are sums of terms of both signs
(policy-gradient loss, actor loss) are compared with an absolute bound 1e-5 x the magnitude of
the summands, stated at each assert.  The measured errors are written to
gpurun_out/parity_measured.json so that profiles/ can quote them.
"""
import json
import os

import numpy as np
import pytest
import torch

from agents_b200 import optimizers
from agents_b200.agents.dqn import dqn_agent
from agents_b200.agents.ppo import ppo_clip_agent
from agents_b200.agents.sac import sac_agent
from agents_b200.networks import actor_distribution_network
from agents_b200.networks import critic_network
from agents_b200.networks import layers as L
from agents_b200.networks import q_network
from agents_b200.networks import tanh_normal_projection_network as tnp
from agents_b200.networks import value_network
from agents_b200.specs import tensor_spec
from agents_b200.trajectories import time_step as ts
from agents_b200.trajectories import trajectory
from oracle import dqn as odqn
from oracle import dqn_torch
from oracle import nn as onn
from oracle import optim as ooptim
from oracle import ppo as oppo
from oracle import sac as osac

pytestmark = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _record(name, **kw):
  path = os.path.join(ROOT, 'gpurun_out', 'parity_measured.json')
  try:
    os.makedirs(os.path.dirname(path), exist_ok=True)
    cur = json.load(open(path)) if os.path.exists(path) else {}
    cur[name] = {k: float(v) for k, v in kw.items()}
    json.dump(cur, open(path, 'w'), indent=1, sort_keys=True)
  except OSError:
    pass


def _rel(got, want):
  return abs(float(got) - float(want)) / max(abs(float(want)), 1e-30)


def _oracle_layers(net):
  out = []
  for l in net.layers:
    if isinstance(l, L.CastScale):
      out.append(dict(kind='cast_scale', divisor=l.divisor))
    elif isinstance(l, L.Conv2D):
      out.append(dict(kind='conv', w=l.kernel.cpu().numpy().copy(), b=l.bias.cpu().numpy().copy(),
                      stride=l.stride, act=l.activation))
    elif isinstance(l, L.Flatten):
      out.append(dict(kind='flatten'))
    elif isinstance(l, L.Dense):
      out.append(dict(kind='dense', w=l.kernel.cpu().numpy().copy(), b=l.bias.cpu().numpy().copy(),
                      act=l.activation))
  return out


def test_config2_dqn_mnih_batch256_train_parity(cuda):
  """agents/dqn/dqn_agent.py:412-579 at examples/dqn/mnih15 shapes: 3 steps."""
  rng = np.random.RandomState(0)
  A, B, T = 6, 256, 2
  obs_spec = tensor_spec.TensorSpec((84, 84, 4), torch.uint8, 'observation')
  act_spec = tensor_spec.BoundedTensorSpec((), torch.int32, 0, A - 1, 'action')
  net = q_network.QNetwork(obs_spec, act_spec, preprocessing_layers=L.CastScale(255.),
                           conv_layer_params=((32, 8, 4), (64, 4, 2), (64, 3, 1)),
                           fc_layer_params=(512,), device=cuda).set_seed(0)
  opt = optimizers.RMSPropOptimizer(2.5e-4, decay=0.95, momentum=0.0, epsilon=1e-5, centered=True)
  agent = dqn_agent.DqnAgent(ts.time_step_spec(obs_spec), act_spec, q_network=net, optimizer=opt,
                             n_step_update=1, target_update_tau=1.0, target_update_period=2,
                             gamma=0.99)
  agent.initialize()
  torch.set_num_threads(min(16, os.cpu_count() or 1))
  orc = dqn_torch.DqnTorchOracle(_oracle_layers(net), target_update_period=2)
  worst_loss, worst_td = 0.0, 0.0
  for step in range(3):
    e = dict(observation=rng.randint(0, 256, size=(B, T, 84, 84, 4)).astype(np.uint8),
             step_type=rng.randint(0, 3, size=(B, T)).astype(np.int32),
             action=rng.randint(0, A, size=(B, T)).astype(np.int32),
             reward=rng.rand(B, T).astype(f32), discount=(rng.rand(B, T) > 0.1).astype(f32))
    d = lambda a: torch.as_tensor(a, device=cuda)
    traj = trajectory.Trajectory(d(e['step_type']), d(e['observation']), d(e['action']), (),
                                 d(e['step_type']), d(e['reward']), d(e['discount']))
    got = agent.train(traj)
    want = orc.train(e)
    worst_loss = max(worst_loss, _rel(got.loss.item(), want))
    np.testing.assert_allclose(got.loss.item(), want, rtol=1e-5)
    assert np.isfinite(got.extra.td_error.cpu().numpy()).all()
  # parameters after 3 RMSProp steps (and one hard target update at step 2)
  worst_p = 0.0
  for v, w in zip(net.variables, orc.q_net.params()):
    w = w.detach().numpy()
    worst_p = max(worst_p, float(np.abs(v.cpu().numpy() - w).max() / max(np.abs(w).max(), 1e-30)))
    np.testing.assert_allclose(v.cpu().numpy(), w, rtol=1e-4, atol=1e-6)
  for v, w in zip(agent._target_q_network.variables, orc.target_net.params()):
    np.testing.assert_allclose(v.cpu().numpy(), w.detach().numpy(), rtol=1e-4, atol=1e-6)
  _record('config2_dqn_mnih_b256', loss_rel=worst_loss, param_rel_to_max=worst_p)
  agent.check_numerics()


def test_dqn_train_parity_all_layers_on_tensor_cores(cuda):
  """5 steps of a conv net whose every layer has >= 16 output channels at batch 32, so conv1 also
  takes the tcgen05 path (numpy oracle, Adam, n-step 2, clipping, Polyak).  conv1 is k4 s4 on the
  28x28x4 uint8 input: stride * C = 16, so the raw-pixel loader of the tensor-core kernel can copy
  its patches in 16-byte chunks (tests/test_gemm_route_gpu.py pins the route)."""
  rng = np.random.RandomState(3)
  A, B, n = 4, 32, 2
  obs_spec = tensor_spec.TensorSpec((28, 28, 4), torch.uint8)
  act_spec = tensor_spec.BoundedTensorSpec((), torch.int32, 0, A - 1)
  net = q_network.QNetwork(obs_spec, act_spec, preprocessing_layers=L.CastScale(255.),
                           conv_layer_params=((16, 4, 4), (32, 3, 1)), fc_layer_params=(64,),
                           device=cuda).set_seed(1)
  agent = dqn_agent.DdqnAgent(ts.time_step_spec(obs_spec), act_spec, q_network=net,
                              optimizer=optimizers.AdamOptimizer(1e-3), n_step_update=n,
                              target_update_tau=0.5, target_update_period=2, gamma=0.99,
                              gradient_clipping=10.0)
  agent.initialize()
  orc = odqn.DqnOracle(onn.Sequential(_oracle_layers(net)), ooptim.AdamTF(1e-3, eps=1e-8), gamma=0.99,
                       n_step_update=n, target_update_tau=0.5, target_update_period=2,
                       gradient_clipping=10.0, ddqn=True)
  worst = 0.0
  for step in range(5):
    e = dict(observation=rng.randint(0, 256, size=(B, n + 1, 28, 28, 4)).astype(np.uint8),
             step_type=rng.randint(0, 3, size=(B, n + 1)).astype(np.int32),
             action=rng.randint(0, A, size=(B, n + 1)).astype(np.int32),
             reward=rng.rand(B, n + 1).astype(f32), discount=(rng.rand(B, n + 1) > 0.1).astype(f32))
    d = lambda a: torch.as_tensor(a, device=cuda)
    traj = trajectory.Trajectory(d(e['step_type']), d(e['observation']), d(e['action']), (),
                                 d(e['step_type']), d(e['reward']), d(e['discount']))
    got = agent.train(traj)
    want = orc.train(e)
    worst = max(worst, _rel(got.loss.item(), want['loss']))
    np.testing.assert_allclose(got.loss.item(), want['loss'], rtol=1e-5)
    np.testing.assert_allclose(got.extra.td_error.cpu().numpy(), want['td_error'], rtol=1e-4, atol=2e-5)
  for v, w in zip(net.variables, orc.q_net.params()):
    np.testing.assert_allclose(v.cpu().numpy(), w, rtol=1e-3, atol=1e-5)
  _record('dqn_conv16_32_b32', loss_rel=worst)


def _mirror_dense(net):
  return onn.Sequential([dict(kind='dense', w=l.kernel.cpu().numpy().copy(), b=l.bias.cpu().numpy().copy(),
                              act=l.activation) for l in net.layers if isinstance(l, L.Dense)])


def test_config3_ppo_200x100_t128_normalizers_on_train_parity(cuda):
  """agents/ppo/ppo_agent.py:834-1076 with the v2 example's nets (200,100) tanh, T=128, GAE,
  normalize_observations=True, normalize_rewards=True; 512 of the 4096 trajectories."""
  rng = np.random.RandomState(11)
  B, T, D, A, epochs = 512, 128, 17, 6, 2
  obs_spec = tensor_spec.TensorSpec((D,), torch.float32, 'observation')
  act_spec = tensor_spec.BoundedTensorSpec((A,), torch.float32, -1.0, 1.0, 'action')
  actor = actor_distribution_network.ActorDistributionNetwork(
      obs_spec, act_spec, fc_layer_params=(200, 100), activation_fn='tanh', device=cuda).set_seed(1)
  value = value_network.ValueNetwork(obs_spec, fc_layer_params=(200, 100), activation_fn='tanh',
                                     device=cuda).set_seed(2)
  agent = ppo_clip_agent.PPOClipAgent(
      ts.time_step_spec(obs_spec), act_spec, optimizer=optimizers.Adam(3e-4), actor_net=actor,
      value_net=value, importance_ratio_clipping=0.2, use_gae=True, lambda_value=0.95,
      discount_factor=0.99, num_epochs=epochs, normalize_observations=True, normalize_rewards=True)
  agent.initialize()
  orc = oppo.PPOOracle(_mirror_dense(actor), actor._std.bias.cpu().numpy().copy(), _mirror_dense(value),
                       -np.ones(A, f32), np.ones(A, f32), ooptim.AdamTF(3e-4, eps=1e-7),
                       num_epochs=epochs, clip_eps=0.2, vf_coef=0.5, gamma=0.99, lam=0.95,
                       normalize_rewards=True, normalize_observations=True, obs_dim=D)
  worst = dict(loss=0.0, ve=0.0, pg_abs=0.0)
  for it in range(2):
    e = dict(observation=(rng.randn(B, T, D) * (1 + it) + .3 * it).astype(f32),
             action=np.clip(rng.randn(B, T, A) * .5, -1, 1).astype(f32),
             loc=(rng.randn(B, T, A) * .2).astype(f32), scale=(rng.rand(B, T, A) * .3 + .5).astype(f32),
             reward=rng.rand(B, T).astype(f32), discount=np.ones((B, T), f32),
             step_type=np.ones((B, T), np.int32), next_step_type=np.ones((B, T), np.int32))
    ends = rng.rand(B, T) < 0.02
    e['next_step_type'][ends] = 2
    e['discount'][ends] = 0
    e['step_type'][:, 1:][ends[:, :-1]] = 2
    want = orc.train(e)[-1]
    d = lambda a: torch.as_tensor(a, device=cuda)
    traj = trajectory.Trajectory(d(e['step_type']), d(e['observation']), d(e['action']),
                                 {'dist_params': {'loc': d(e['loc']), 'scale': d(e['scale'])}},
                                 d(e['next_step_type']), d(e['reward']), d(e['discount']))
    got = agent.train(traj)
    worst['loss'] = max(worst['loss'], _rel(got.loss.item(), want['loss']))
    worst['ve'] = max(worst['ve'], _rel(got.extra.value_estimation_loss.item(), want['ve']))
    worst['pg_abs'] = max(worst['pg_abs'], abs(got.extra.policy_gradient_loss.item() - want['pg']))
    np.testing.assert_allclose(got.loss.item(), want['loss'], rtol=1e-5)
    np.testing.assert_allclose(got.extra.value_estimation_loss.item(), want['ve'], rtol=1e-5)
    # the surrogate is a mean of ratio * A_hat terms of both signs with |A_hat| ~ 1 (normalised
    # advantages): 1e-5 of the summand magnitude, not of the near-cancelling sum
    np.testing.assert_allclose(got.extra.policy_gradient_loss.item(), want['pg'], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(got.extra.clip_fraction.item(), want['clip_fraction'], atol=4.0 / (B * T))
  cnt, avg, m2, _ = [t.cpu().numpy() for t in agent._observation_normalizer.variables]
  np.testing.assert_allclose(cnt, orc.obs_normalizer.count, rtol=1e-6)
  np.testing.assert_allclose(avg, orc.obs_normalizer.avg, rtol=1e-4, atol=1e-5)
  np.testing.assert_allclose(m2, orc.obs_normalizer.m2, rtol=1e-4)
  for v, w in zip(actor.variables + value.variables, orc.actor.params() + [orc.std_bias] + orc.value.params()):
    np.testing.assert_allclose(v.cpu().numpy(), w, rtol=2e-3, atol=2e-5)
  _record('config3_ppo_512x128', **worst)
  agent.check_numerics()


def test_config4_sac_256x256_batch1024_train_parity(cuda):
  """agents/sac/sac_agent.py:314-410 at the haarnoja18 example's sizes: 3 steps, supplied noise."""
  rng = np.random.RandomState(5)
  D, A, B = 17, 6, 1024
  obs_spec = tensor_spec.TensorSpec((D,), torch.float32, 'observation')
  act_spec = tensor_spec.BoundedTensorSpec((A,), torch.float32, -1.0, 1.0, 'action')
  actor = tnp.TanhNormalActorNetwork(obs_spec, act_spec, fc_layer_params=(256, 256), device=cuda).set_seed(1)
  critic = critic_network.CriticNetwork((obs_spec, act_spec), joint_fc_layer_params=(256, 256),
                                        device=cuda).set_seed(2)
  agent = sac_agent.SacAgent(ts.time_step_spec(obs_spec), act_spec, critic_network=critic,
                             actor_network=actor, actor_optimizer=optimizers.Adam(3e-4),
                             critic_optimizer=optimizers.Adam(3e-4), alpha_optimizer=optimizers.Adam(3e-4),
                             target_update_tau=0.005, target_update_period=1, gamma=0.99,
                             reward_scale_factor=0.1)
  agent.initialize()
  orc = osac.SacOracle(_mirror_dense(actor), _mirror_dense(agent._critic_network_1),
                       _mirror_dense(agent._critic_network_2), -np.ones(A, f32), np.ones(A, f32),
                       ooptim.AdamTF(3e-4, eps=1e-7), ooptim.AdamTF(3e-4, eps=1e-7),
                       ooptim.AdamTF(3e-4, eps=1e-7), gamma=0.99, reward_scale=0.1, tau=0.005)
  worst = dict(critic=0.0, actor_abs=0.0, alpha_abs=0.0)
  for step in range(3):
    e = dict(observation=rng.randn(B, 2, D).astype(f32), action=(rng.rand(B, 2, A) * 2 - 1).astype(f32),
             reward=rng.rand(B, 2).astype(f32), discount=(rng.rand(B, 2) > .05).astype(f32))
    noise = [rng.randn(B, A).astype(f32) for _ in range(3)]
    want = orc.train(e, *noise)
    d = lambda a: torch.as_tensor(a, device=cuda)
    traj = trajectory.Trajectory(torch.ones(B, 2, dtype=torch.int32, device=cuda), d(e['observation']),
                                 d(e['action']), (), torch.ones(B, 2, dtype=torch.int32, device=cuda),
                                 d(e['reward']), d(e['discount']))
    got = agent.train(traj, noise=noise)
    worst['critic'] = max(worst['critic'], _rel(got.extra.critic_loss.item(), want['critic_loss']))
    worst['actor_abs'] = max(worst['actor_abs'], abs(got.extra.actor_loss.item() - want['actor_loss']))
    worst['alpha_abs'] = max(worst['alpha_abs'], abs(got.extra.alpha_loss.item() - want['alpha_loss']))
    np.testing.assert_allclose(got.extra.critic_loss.item(), want['critic_loss'], rtol=1e-5)
    # actor / alpha losses are means of log-prob (|.| ~ 5) and Q terms of both signs
    np.testing.assert_allclose(got.extra.actor_loss.item(), want['actor_loss'], rtol=1e-5, atol=5e-5)
    np.testing.assert_allclose(got.extra.alpha_loss.item(), want['alpha_loss'], rtol=1e-5, atol=5e-5)
    np.testing.assert_allclose(got.loss.item(), want['loss'], rtol=1e-5, atol=5e-5)
  # Adam divides by sqrt(v): where a gradient element is ~0 (dead ReLU paths) a 1e-9 difference
  # in g moves the parameter by up to lr per step, so parameters are compared as "all but a
  # vanishing fraction within 1e-3 relative, none further than steps * lr" (measured on B200:
  # 8 of 65 536 actor weights beyond the tight bound, max 5.2e-4)
  bad, total, worst_abs = 0, 0, 0.0
  for v, w in zip(actor.variables, orc.actor.params()):
    g = v.cpu().numpy()
    bad += int((np.abs(g - w) > 1e-5 + 1e-3 * np.abs(w)).sum())
    total += w.size
    worst_abs = max(worst_abs, float(np.abs(g - w).max()))
  assert bad <= 1e-3 * total and worst_abs <= 3 * 3e-4 * 1.05, (bad, total, worst_abs)
  # the target moves by tau * (critic - target) per step, so the same Adam outliers show up scaled
  # by tau (measured: 1 of 5888 first-layer weights off by 8.2e-6)
  for v, w in zip(agent._target_critic_network_1.variables, orc.t1.params()):
    np.testing.assert_allclose(v.cpu().numpy(), w, rtol=1e-4, atol=2e-5)
  worst['actor_param_outliers'] = bad
  worst['actor_param_max_abs'] = worst_abs
  _record('config4_sac_b1024', **worst)
  agent.check_numerics()
