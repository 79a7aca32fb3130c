"""train.Learner on the GPU: DQN through buffer -> dataset -> Learner.run, checkpoints, and (when
>= 2 GPUs are visible) NCCL data-parallel parity against a single replica via torchrun."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

from agents_b200 import optimizers
from agents_b200.agents.dqn import dqn_agent
from agents_b200.drivers import dynamic_step_driver
from agents_b200.environments import random_tf_environment
from agents_b200.networks import layers as L
from agents_b200.networks import sequential
from agents_b200.replay_buffers import tf_uniform_replay_buffer as rb_mod
from agents_b200.train import learner as learner_lib
from agents_b200.train.utils import train_utils

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup(cuda, seed=0):
  env = random_tf_environment.CartPoleTFEnvironment(batch_size=4, seed=seed, device=cuda, action_dtype=torch.int32)
  tss, act_spec = env.time_step_spec(), env.action_spec()
  net = sequential.Sequential([L.Dense(32, activation='relu'), L.Dense(2)], input_spec=tss.observation,
                              device=cuda).set_seed(seed)
  train_step = train_utils.create_train_step(cuda)
  agent = dqn_agent.DqnAgent(tss, act_spec, q_network=net, optimizer=optimizers.AdamOptimizer(1e-3), gamma=0.99,
                             target_update_period=3, train_step_counter=train_step)
  agent.initialize()
  rb = rb_mod.TFUniformReplayBuffer(agent.collect_data_spec, batch_size=4, max_length=256, device=cuda, seed=seed)
  dynamic_step_driver.DynamicStepDriver(env, agent.collect_policy, observers=[rb.add_batch], num_steps=200).run()
  return agent, rb, train_step


def test_learner_run_and_checkpoint(cuda):
  root = tempfile.mkdtemp()
  agent, rb, train_step = _setup(cuda)
  lrn = learner_lib.Learner(root, train_step, agent,
                            experience_dataset_fn=lambda: rb.as_dataset(sample_batch_size=32, num_steps=2),
                            checkpoint_interval=4)
  info = lrn.run(iterations=5)
  assert np.isfinite(info.loss.item()) and int(train_step.item()) == 5
  ckpts = os.listdir(os.path.join(root, 'train', 'checkpoints'))
  assert len(ckpts) == 1
  agent2, rb2, train_step2 = _setup(cuda, seed=1)
  learner_lib.Learner(root, train_step2, agent2,
                      experience_dataset_fn=lambda: rb2.as_dataset(sample_batch_size=32, num_steps=2),
                      checkpoint_interval=4)
  assert int(train_step2.item()) == 5
  assert torch.equal(agent._q_network.flat_params, agent2._q_network.flat_params)
  opt1 = list(agent._optimizer._slots.values())[0]
  assert int(opt1['step'][0].item()) == 5


def test_checkpointer_resumes_ring_agent_and_optimizer(cuda, tmp_path):
  """common.Checkpointer (utils/common.py:1045-1100) over agent + replay buffer + global step: a
  restored run samples the same rows and produces bit-identical losses as the original."""
  from agents_b200.utils import common
  agent, rb, train_step = _setup(cuda)
  for _ in range(3):
    exp, _ = rb.get_next(sample_batch_size=16, num_steps=2)
    agent.train(exp)
  ck = common.Checkpointer(str(tmp_path), max_to_keep=1, agent=agent, replay_buffer=rb,
                           global_step=train_step)
  assert not ck.checkpoint_exists
  ck.save(train_step)
  want = []
  for _ in range(3):
    exp, info = rb.get_next(sample_batch_size=16, num_steps=2)
    want.append((info.ids.cpu().numpy().copy(), float(agent.train(exp).loss.item())))
  agent2, rb2, train_step2 = _setup(cuda, seed=1)                  # different weights and data
  ck2 = common.Checkpointer(str(tmp_path), max_to_keep=1, agent=agent2, replay_buffer=rb2,
                            global_step=train_step2)
  assert ck2.checkpoint_exists and ck2.initialize_or_restore()
  assert int(train_step2.item()) == 3 and rb2.num_frames() == rb.num_frames()
  for ids, loss in want:
    exp, info = rb2.get_next(sample_batch_size=16, num_steps=2)
    np.testing.assert_array_equal(info.ids.cpu().numpy(), ids)
    assert float(agent2.train(exp).loss.item()) == loss


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_nccl_data_parallel_parity():
  cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
         '--master-addr', '127.0.0.1', '--master-port', '29517', os.path.join(ROOT, 'tests', 'dist_parity_main.py')]
  out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
  assert 'DIST_PARITY_OK' in out.stdout
