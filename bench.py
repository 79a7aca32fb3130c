"""bench.py — train steps/sec (DQN Atari-shape, batch 256) on N B200s, replay GB/s.

Workload (BASELINE.json configs[1]): synthetic Atari-shape observations 84x84x4 uint8, a
1 048 576-slot TFUniformReplayBuffer (256 segments x 4096) per GPU, sample batch 256 x T=2,
Mnih'15 Q-network, Huber loss, centered RMSProp (examples/dqn/mnih15 config), gamma 0.99, hard
target update every 2500 steps.  One "step" = get_next(256, 2) + DqnAgent.train(experience).

  value        steps/s with the ring resident in HBM; the step is replayed as ONE CUDA graph.
               `--steps K` steps are timed `--repeats R` times (default once; each block
               bracketed by barrier + synchronize, CUDA events, max over ranks); value is the
               MEDIAN block.  The e2e arm and the update-only roofline also time K steps.
  e2e          the same step through the public API with HOST buffers: every step copies one
               driver step of collected frames (256 x 28 244 B) from pinned host memory,
               add_batch, get_next, train, and reads that step's loss back (the read of step
               i-1 overlaps step i: pinned 4-byte slots + events).
  parity       before timing, 3 train steps on the sampled batches are replayed by the CPU
               restatement (oracle/dqn_torch.py, same initial weights) and the losses compared.
  roofline     the update's GEMM/conv work against the measured tensor peak; roofline_gather:
               the replay gather kernel against measured HBM GB/s.
  cpu_baseline the torch-CPU restatement of the reference train step on the host cores
               (TensorFlow is not installable here, BASELINE.md §3): 1 M-slot host ring when RAM
               allows, physical-core thread count, median of 3 blocks.
  ppo_update / sac_step / cartpole_iter / gather_sweep   BASELINE configs 3 / 4 / 1 / 5
               (profiles/configs.py); under torchrun they are sharded over the ranks.
  dp_parity    (N > 1) N replicas on shards vs one replica on the whole batch.
The main line is complete before the extra configs and the CPU arm start; they only add keys, and
a watchdog (`--extras-timeout`, 600 s) prints the line without them should one of them hang.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step computed as
DIR/<name>.npy (float32 / float64): its loss, td_loss and td_error, the Q-network and target-network
parameters after the update, and the batch it trained on (ids, probabilities, the scalar leaves and
a fixed seeded sample of the observation bytes).  Every input is seeded, so two builds run with the
same arguments can be compared output for output.

`--impl reference` times that CPU restatement alone (the reference arm of the project).
N>1 (torchrun): one process per GPU, each with its own 1M-slot ring shard and a local batch of
256; gradients are SUM-all-reduced (NCCL) every step, loss is divided by the global batch
(utils/common.py:1465-1467).  value = batch-256-equivalent train steps/s of the whole job
(weak scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

ROW_BYTES = 4 + 28224 + 4 + 4 + 4 + 4          # SURVEY.md §8: Atari-shape Trajectory row
A = 6
B, T = 256, 2
B_ENV, L = 256, 4096
CONV = ((32, 8, 4), (64, 4, 2), (64, 3, 1))
FC = (512,)
# Mnih'15 net forward = 9.35 M MAC/sample (SURVEY §8d); step = fwd(s0) + fwd_target(sn) + bwd(2x)
FLOPS_PER_STEP = 4 * 2 * 9.35e6 * B
GATHER_BYTES = 2 * B * T * ROW_BYTES + 8 * B * T
WORKLOAD = (f'DQN synthetic Atari-shape obs 84x84x4 uint8, 1M-slot replay ({B_ENV}x{L}), '
            f'batch {B}, T={T}, Mnih15 net, Huber, centered RMSProp')


def _peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    d = json.load(open(p))
    return dict(hbm=d['hbm_gbs'], tensor_burst=d['bf16_tflops'],
                tensor=d.get('bf16_tflops_sustained', d['bf16_tflops']), src='measured')
  return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, src='fallback')


def _mnih_layers(rng):
  """numpy parameter dicts of the Mnih'15 net (for the CPU arm)."""
  layers = [dict(kind='cast_scale', divisor=255.0)]
  c_in, hw = 4, 84
  for f, k, s in CONV:
    fan = k * k * c_in
    layers.append(dict(kind='conv', w=(rng.randn(k, k, c_in, f) * np.sqrt(2.0 / fan)).astype(np.float32),
                       b=np.zeros(f, np.float32), stride=s, act='relu'))
    c_in, hw = f, (hw - k) // s + 1
  layers.append(dict(kind='flatten'))
  n_in = hw * hw * c_in
  for u in FC:
    layers.append(dict(kind='dense', w=(rng.randn(n_in, u) * np.sqrt(2.0 / n_in)).astype(np.float32),
                       b=np.zeros(u, np.float32), act='relu'))
    n_in = u
  layers.append(dict(kind='dense', w=(rng.rand(n_in, A) * 0.06 - 0.03).astype(np.float32),
                     b=np.full(A, -0.2, np.float32), act=None))
  return layers


def _physical_cores():
  """Distinct (physical id, core id) pairs of /proc/cpuinfo; falls back to half the logical CPUs."""
  try:
    pairs, phys = set(), None
    for line in open('/proc/cpuinfo'):
      if line.startswith('physical id'):
        phys = line.split(':')[1].strip()
      elif line.startswith('core id'):
        pairs.add((phys, line.split(':')[1].strip()))
    if pairs:
      return len(pairs)
  except OSError:
    pass
  return max(1, (os.cpu_count() or 2) // 2)


def _host_ram_gb():
  try:
    for line in open('/proc/meminfo'):
      if line.startswith('MemAvailable'):
        return int(line.split()[1]) / 1e6
  except OSError:
    pass
  return 0.0


class CpuArm(object):
  """The CPU restatement of one step: numpy ring gather (oracle/replay.py) + torch-CPU train
  (oracle/dqn_torch.py).  1 M-slot ring (256 x 4096, 29.6 GB) when the host has >= 48 GB
  available, else the largest power-of-two ring that fits in a quarter of it."""

  def __init__(self, seed=0):
    import torch
    from oracle import dqn_torch
    from oracle import replay as oreplay
    rng = np.random.RandomState(seed)
    avail = _host_ram_gb()
    b_env, l = B_ENV, L
    while b_env * l * ROW_BYTES / 1e9 > max(avail - 18.0, avail * 0.25) and l > 64:
      l //= 2
    self.b_env, self.l = b_env, l
    shapes = [(), (84, 84, 4), (), (), (), ()]
    dtypes = [np.int32, np.uint8, np.int32, np.int32, np.float32, np.float32]
    self.ring = oreplay.UniformReplayOracle(shapes, dtypes, b_env, l, seed=seed)
    obs = self.ring.storage[1]
    block = rng.randint(0, 256, size=(min(2048, obs.shape[0]),) + obs.shape[1:], dtype=np.uint8)
    for i in range(0, obs.shape[0], block.shape[0]):           # tile a 58 MB random block
      n = min(block.shape[0], obs.shape[0] - i)
      obs[i:i + n] = block[:n]
    cap = self.ring.capacity
    self.ring.storage[0][...] = rng.randint(0, 3, size=cap)
    self.ring.storage[2][...] = rng.randint(0, A, size=cap)
    self.ring.storage[4][...] = rng.rand(cap)
    self.ring.storage[5][...] = (rng.rand(cap) > 0.1)
    self.ring.last_id = 2 * l + 17
    self.agent = dqn_torch.DqnTorchOracle(_mnih_layers(rng))
    self.torch = torch
    self.threads = min(_physical_cores(), os.cpu_count() or 1)
    torch.set_num_threads(self.threads)

  def step(self):
    data, _, _, _ = self.ring.get_next(B, T)
    return self.agent.train(dict(step_type=data[0], observation=data[1], action=data[2],
                                 reward=data[4], discount=data[5]))

  def time_block(self, steps):
    t0 = time.perf_counter()
    for _ in range(steps):
      self.step()
    return steps / (time.perf_counter() - t0)

  def measure(self, steps, warmup, blocks=3):
    """Returns (median steps/s at the FASTEST thread count of a short sweep, sweep dict, description).

    More threads are not faster for this small-batch workload (oneDNN conv on 64 cores ran at a
    third of its 16-thread rate on the round-2 box), so the arm first times one short block at
    each of {physical cores, half of them, 32, 16, 8} and then takes the median of `blocks` blocks
    at the best count: the CPU number the GPU is compared with is the strongest one found."""
    for _ in range(max(3, warmup)):
      self.step()
    phys = self.threads
    sweep = {}
    for nt in sorted({phys, max(1, phys // 2), 32, 16, 8}):
      if 1 <= nt <= (os.cpu_count() or 1):
        self.torch.set_num_threads(nt)
        self.step()
        sweep[str(nt)] = self.time_block(max(2, steps // 2))
    best = int(max(sweep, key=lambda k: sweep[k]))
    self.threads = best
    self.torch.set_num_threads(best)
    self.step()
    sps = sorted(self.time_block(steps) for _ in range(blocks))
    med = sps[len(sps) // 2]
    sample = (f'{blocks} blocks x {steps} train steps after {max(3, warmup)} warm-up steps (batch {B}, '
              f'T={T}, Mnih15 net, torch-CPU restatement, {self.b_env}x{self.l}-slot host ring); '
              f'{best} threads = fastest of the sweep {sorted(int(k) for k in sweep)} on {phys} physical '
              f'cores; median block')
    return med, sweep, sample


class ClockSampler(object):
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    self.index = index
    self.proc = None
    self.path = f'/tmp/b200rl_clocks_{os.getpid()}.csv'

  def start(self):
    try:
      self.f = open(self.path, 'w')
      self.proc = subprocess.Popen(
          ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '50',
           '-i', str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
    except Exception:
      self.proc = None

  def stop(self):
    out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
    if self.proc is None:
      return out
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      self.proc.kill()
    self.f.close()
    sm, mx, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for line in open(self.path):
      p = [x.strip() for x in line.split(',')]
      if len(p) < 9:
        continue
      try:
        sm.append(float(p[1]))
        mx.append(float(p[2]))
      except ValueError:
        continue
      for n, v in zip(names, p[5:9]):
        if v.lower().startswith('active'):
          reasons.add(n)
    if sm:
      out = dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                 samples=len(sm))
    try:
      os.remove(self.path)
    except OSError:
      pass
    return out


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  steps = args.steps
  warm = max(3, args.warmup)
  arm = CpuArm()
  sps, sweep, sample = arm.measure(steps, warm)
  line = dict(
      impl='reference', metric='train steps/sec (DQN Atari-shape, batch 256)', value=sps,
      unit='steps/s', n_gpus=args.gpus, steps=steps, warmup=warm,
      ms_per_step=1000.0 / sps, higher_is_better=True, scaling='weak', vs_baseline=None,
      dtype='f32', data='synthetic',
      config=dict(workload=WORKLOAD, global_batch=B, per_gpu_batch=B, num_actions=A,
                  host_ring=f'{arm.b_env}x{arm.l}',
                  parallelism='cpu (host cores of the box, rank 0 only)'),
      cpu_baseline=dict(value=sps, unit='steps/s', cores=arm.threads, kind='port', sample=sample,
                        other_thread_counts=sweep, logical_cpus=os.cpu_count()),
      e2e=dict(value=sps, unit='steps/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
  print(json.dumps(line), flush=True)


def _oracle_layers(net, Ly):
  layers = [dict(kind='cast_scale', divisor=255.0)]
  for l in net.layers:
    if isinstance(l, Ly.Conv2D):
      layers.append(dict(kind='conv', w=l.kernel.cpu().numpy().copy(), b=l.bias.cpu().numpy().copy(),
                         stride=l.stride, act=l.activation))
    elif isinstance(l, Ly.Flatten):
      layers.append(dict(kind='flatten'))
    elif isinstance(l, Ly.Dense):
      layers.append(dict(kind='dense', w=l.kernel.cpu().numpy().copy(), b=l.bias.cpu().numpy().copy(),
                         act=l.activation))
  return layers


OBS_SAMPLE = 1 << 16        # observation bytes of the trained batch written by --dump-outputs


def dump_outputs(out_dir, loss_info, batch, net, target_net):
  """Writes the last timed step's results as out_dir/<name>.npy (float32, or float64 for the
  int64 ids and the integer leaves so that they stay exact)."""
  exp, info = batch
  tensors = dict(loss=loss_info.loss, td_loss=loss_info.extra.td_loss,
                 td_error=loss_info.extra.td_error, q_network_params=net.flat_params,
                 target_q_network_params=target_net.flat_params, ids=info.ids,
                 probabilities=info.probabilities)
  for name in ('step_type', 'action', 'next_step_type', 'reward', 'discount'):
    tensors[name] = getattr(exp, name)
  arrays = {k: t.detach().cpu().numpy() for k, t in tensors.items()}
  obs = exp.observation.cpu().numpy().reshape(-1)
  pick = np.sort(np.random.RandomState(0).choice(obs.size, min(OBS_SAMPLE, obs.size), replace=False))
  arrays['observation_sample'] = obs[pick]
  arrays = {k: a.astype(np.float32 if a.dtype in (np.float32, np.uint8) else np.float64)
            for k, a in arrays.items()}
  total = sum(a.nbytes for a in arrays.values())
  assert total <= 64 << 20, f'--dump-outputs would write {total} bytes'
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), a)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=200, help='train steps in each timed loop')
  ap.add_argument('--warmup', type=int, default=10)
  ap.add_argument('--repeats', type=int, default=1,
                  help='timed blocks of --steps steps for `value` (its median block)')
  ap.add_argument('--impl', default='b200')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-graph', action='store_true')
  ap.add_argument('--no-extra', action='store_true', help='skip configs 1/3/4/5 and dp_parity')
  ap.add_argument('--extras-timeout', type=float, default=600.0,
                  help='seconds the extra configs + CPU arm may take before the line is printed without them')
  ap.add_argument('--no-prefetch', action='store_true',
                  help='sample and train back to back on one stream (default: the sample of step '
                       'i+1 runs on a side stream beside train(i), like dataset.prefetch(1))')
  ap.add_argument('--ncu-step', action='store_true',
                  help='after warm-up run ONE un-captured step between cudaProfilerStart/Stop and '
                       'exit (target of `ncu --profile-from-start off`; prints no bench value)')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write what the last timed step computed to DIR/<name>.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be >= 1')
  if args.impl == 'reference':
    return run_reference(args)

  import torch
  import torch.distributed as dist
  from agents_b200 import _lib
  from agents_b200 import optimizers
  from agents_b200.agents.dqn import dqn_agent
  from agents_b200.networks import layers as Ly
  from agents_b200.networks import q_network
  from agents_b200.replay_buffers import tf_uniform_replay_buffer as rb_mod
  from agents_b200.specs import tensor_spec
  from agents_b200.train.utils import strategy_utils
  from agents_b200.trajectories import time_step as ts
  from agents_b200.trajectories import trajectory
  from agents_b200.utils import common

  if not torch.cuda.is_available():
    raise SystemExit('bench.py needs a CUDA device: the hot path has no CPU fallback.')
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  if world > 1:
    strategy_utils.configure_nccl_env()
    dist.init_process_group('nccl', device_id=dev)
  strategy = strategy_utils.get_strategy()
  W = max(args.warmup, 3)
  K = args.steps
  R = max(1, args.repeats)
  peaks = _peaks()
  extra = {}

  def guarded(name, fn):
    try:
      extra[name] = fn()
      torch.cuda.synchronize()
    except Exception as e:  # pylint: disable=broad-except
      extra[name] = dict(error=f'{type(e).__name__}: {e}')
      sys.stderr.write(f'[rank {rank}] {name} failed: {type(e).__name__}: {e}\n')

  # ---- data-parallel parity first (small, eager; uses the process group before any graph) -------
  if world > 1 and not args.no_extra:
    from profiles import configs
    guarded('dp_parity', lambda: configs.dp_parity(strategy, dev))

  # ---- build the workload ---------------------------------------------------------------------
  obs_spec = tensor_spec.TensorSpec((84, 84, 4), torch.uint8, 'observation')
  act_spec = tensor_spec.BoundedTensorSpec((), torch.int32, 0, A - 1, 'action')
  net = q_network.QNetwork(obs_spec, act_spec, preprocessing_layers=Ly.CastScale(255.),
                           conv_layer_params=CONV, fc_layer_params=FC, device=dev).set_seed(0)
  opt = optimizers.RMSPropOptimizer(2.5e-4, decay=0.95, momentum=0.0, epsilon=1e-5, centered=True)
  agent = dqn_agent.DqnAgent(ts.time_step_spec(obs_spec), act_spec, q_network=net, optimizer=opt,
                             epsilon_greedy=0.01, n_step_update=1, target_update_tau=1.0,
                             target_update_period=2500, gamma=0.99, seed=0x5eed0000 + rank)
  agent.initialize()
  if world > 1:
    agent.replicas = world
    agent._grad_sync = lambda g: dist.all_reduce(g, op=dist.ReduceOp.SUM)
    dist.broadcast(net.flat_params, 0)
    dist.broadcast(agent._target_q_network.flat_params, 0)
  spec = agent.collect_data_spec
  rb = rb_mod.TFUniformReplayBuffer(spec, batch_size=B_ENV, max_length=L, device=dev,
                                    seed=0x5eed0000 + rank)
  g = torch.Generator(device=dev).manual_seed(1234 + rank)
  st_store, obs_store, act_store, nst_store, rew_store, disc_store = rb._data_table.variables()
  cap = B_ENV * L
  chunk = 1 << 15
  for i in range(0, cap, chunk):               # fill the ring in place (28 GB of random frames)
    obs_store[i:i + chunk].view(-1).view(torch.int64).random_(generator=g)
  st_store.copy_(torch.randint(0, 3, (cap,), device=dev, generator=g, dtype=torch.int32))
  nst_store.copy_(torch.randint(0, 3, (cap,), device=dev, generator=g, dtype=torch.int32))
  act_store.copy_(torch.randint(0, A, (cap,), device=dev, generator=g, dtype=torch.int32))
  rew_store.copy_(torch.rand(cap, device=dev, generator=g))
  disc_store.copy_((torch.rand(cap, device=dev, generator=g) > 0.1).float())
  last_id = 2 * L + 77
  pos = torch.arange(cap, device=dev, dtype=torch.int64) % L
  rb._id_table.variables()[0].copy_(torch.where(pos <= last_id % L, last_id - last_id % L + pos,
                                                last_id - last_id % L - L + pos))
  rb._last_id.fill_(last_id)
  rb._last_id_host = last_id

  # ---- parity at the bench config: 3 steps, GPU vs the CPU restatement on the same batches ------
  parity = None
  cpu_arm_layers = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    from oracle import dqn_torch
    torch.set_num_threads(min(_physical_cores(), os.cpu_count() or 1))
    orc = dqn_torch.DqnTorchOracle(_oracle_layers(net, Ly))
    rels, last = [], None
    for _ in range(3):
      exp, _ = rb.get_next(sample_batch_size=B, num_steps=T)
      got = float(agent.train(exp).loss.item())
      want = orc.train(dict(step_type=exp.step_type.cpu().numpy(), observation=exp.observation.cpu().numpy(),
                            action=exp.action.cpu().numpy(), reward=exp.reward.cpu().numpy(),
                            discount=exp.discount.cpu().numpy()))
      rels.append(abs(got - want) / max(abs(want), 1e-12))
      last = (got, want)
    parity = dict(steps=3, max_rel_loss_err=max(rels), tolerance=1e-5, gpu_loss=last[0],
                  oracle_loss=last[1], oracle='oracle/dqn_torch.py (torch CPU fp32, same initial weights, '
                  'same sampled batches)', ok=bool(max(rels) <= 1e-5))
    if not parity['ok']:
      sys.stderr.write(f'PARITY FAILED at the bench config: {parity}\n')

  # Input pipeline.  The reference's examples train from `replay_buffer.as_dataset(...).prefetch(n)`
  # (agents/dqn/examples/v2/train_eval.py:226-232): the next batch is produced while the current
  # one trains.  Here: two sample buffers; step i trains on buffer i & 1 while the sampler fills
  # the other one on a side stream (same Philox draw order as back-to-back calls).  Every step
  # still contains one sample and one train.  A step returns (LossInfo, the (experience,
  # BufferInfo) batch it trained on).
  prefetch = not args.no_prefetch
  side_stream = torch.cuda.Stream(device=dev)
  sample_bufs = [rb.get_next(sample_batch_size=B, num_steps=T) for _ in range(2)]
  step_no = [0]

  def pipelined(slot):
    def body():
      main = torch.cuda.current_stream()
      side_stream.wait_stream(main)
      with torch.cuda.stream(side_stream):
        rb.get_next(sample_batch_size=B, num_steps=T, out=sample_bufs[slot ^ 1])
      loss_info = agent.train(sample_bufs[slot][0])
      main.wait_stream(side_stream)
      return loss_info, sample_bufs[slot]
    return body

  def serial_step():
    batch = rb.get_next(sample_batch_size=B, num_steps=T)
    return agent.train(batch[0]), batch

  bodies = [pipelined(0), pipelined(1)]

  def step():
    if not prefetch:
      return serial_step()
    step_no[0] += 1
    return bodies[(step_no[0] - 1) & 1]()

  def sync_all():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  # launches of OUR kernels per step (counted on one eager step)
  step()
  torch.cuda.synchronize()
  c0 = _lib.launch_count()
  step()
  torch.cuda.synchronize()
  launches_per_step = _lib.launch_count() - c0

  use_graph = not args.no_graph
  if use_graph and prefetch:
    graphs = [common.function(b, warmup=1) for b in bodies]

    def fn():
      step_no[0] += 1
      return graphs[(step_no[0] - 1) & 1]()
  else:
    fn = common.function(step, warmup=1) if use_graph else step
  fn()                                   # eager warm-up call (sizes workspaces)
  if use_graph and prefetch:
    fn()                                 # ... of the second buffer's graph as well
  ok = 1
  try:
    fn()                                 # capture + first replay
    if use_graph and prefetch:
      fn()
  except Exception as e:  # a step that cannot be captured on this stack -> eager
    if not use_graph:
      raise
    sys.stderr.write(f'[rank {rank}] CUDA-graph capture failed ({type(e).__name__}: {e})\n')
    ok = 0
    torch.cuda.synchronize()
    step()                               # keeps the collective count equal to a successful rank's
  if world > 1 and use_graph:            # all ranks must agree on graph vs eager
    flag = torch.tensor([ok], device=dev, dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = int(flag.item())
  if use_graph and not ok:
    use_graph = False
    fn = step
  for _ in range(W):
    fn()
  sync_all()
  if args.ncu_step:
    torch.cuda.cudart().cudaProfilerStart()
    step()
    torch.cuda.synchronize()
    torch.cuda.cudart().cudaProfilerStop()
    if rank == 0:
      print(json.dumps({'ncu_step': True, 'launches_per_step': launches_per_step}))
    return

  # ---- timed region: R blocks of K steps, CUDA events, max over ranks, median block -------------
  clocks = ClockSampler(local_rank)
  clocks.start()
  block_ms = []
  t_wall0 = time.perf_counter()
  for _ in range(R):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(K):
      loss_info, batch = fn()
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    if world > 1:
      t = torch.tensor([ms], device=dev, dtype=torch.float64)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t.item())
    block_ms.append(ms)
  # graph outputs are overwritten by the next replay: read the last timed step's results now
  final_loss = float(loss_info.loss.item())
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, loss_info, batch, net, agent._target_q_network)
  # keep the sampler running over a load of at least ~1.5 s so that it sees the step's clocks
  while time.perf_counter() - t_wall0 < 1.5:
    for _ in range(K):
      fn()
    torch.cuda.synchronize()
  clk = clocks.stop()
  ms = float(np.median(block_ms))
  agent.check_numerics()
  steps_per_s = K / (ms / 1000.0)
  value = steps_per_s * world                  # batch-256-equivalent steps/s of the whole job

  # ---- per-kernel timing for the rooflines (CUDA events on the launch stream) -------------------
  # 20 gather launches (fresh Philox rows, distinct outputs) captured in one graph so that the
  # events bracket kernel time, not Python launch overhead; replayed 10x.
  n_g, reps = 20, 10
  outs = []
  for _ in range(3):
    rb.get_next(sample_batch_size=B, num_steps=T)
  torch.cuda.synchronize()
  gg = torch.cuda.CUDAGraph()
  with torch.cuda.graph(gg):
    for _ in range(n_g):
      outs.append(rb.get_next(sample_batch_size=B, num_steps=T))
  gg.replay()
  torch.cuda.synchronize()
  ge0, ge1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ge0.record()
  for _ in range(reps):
    gg.replay()
  ge1.record()
  torch.cuda.synchronize()
  gather_ms = ge0.elapsed_time(ge1) / (n_g * reps)
  del outs, gg
  exp, _ = rb.get_next(sample_batch_size=B, num_steps=T)
  n_u = K
  ue0, ue1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  # the update alone, replayed from its own graph so that the events bracket GPU time
  train_only = common.function(lambda: agent.train(exp), warmup=1) if use_graph else (
      lambda: agent.train(exp))
  for _ in range(3):
    train_only()
  torch.cuda.synchronize()
  ue0.record()
  for _ in range(n_u):
    train_only()
  ue1.record()
  torch.cuda.synchronize()
  update_ms = ue0.elapsed_time(ue1) / n_u
  traffic = {}
  tp = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
  if os.path.exists(tp):
    traffic = json.load(open(tp))
  gather_gbs = GATHER_BYTES / (gather_ms * 1e-3) / 1e9
  update_tfs = FLOPS_PER_STEP / (update_ms * 1e-3) / 1e12

  # ---- e2e: host buffers in, loss out, every step -----------------------------------------------
  Ke = K
  gh = torch.Generator().manual_seed(4321 + rank)
  host = [torch.randint(0, 3, (B_ENV,), dtype=torch.int32, generator=gh).pin_memory(),
          torch.randint(0, 256, (B_ENV, 84, 84, 4), dtype=torch.uint8, generator=gh).pin_memory(),
          torch.randint(0, A, (B_ENV,), dtype=torch.int32, generator=gh).pin_memory(),
          torch.randint(0, 3, (B_ENV,), dtype=torch.int32, generator=gh).pin_memory(),
          torch.rand(B_ENV, generator=gh).pin_memory(), torch.ones(B_ENV).pin_memory()]
  h2d = sum(t.numel() * t.element_size() for t in host)

  # Double-buffered upload: the pinned->device copy of step i+1's frames runs on a copy stream
  # while step i trains.  The loss of every step is copied into its own pinned 4-byte slot right
  # after the step (asynchronous D2H on the main stream + an event); the host reads step i-1's
  # slot while step i runs, so the read-back never drains the pipeline and every loss is read.
  copy_stream = torch.cuda.Stream(device=dev)
  main_stream = torch.cuda.current_stream()
  staged = [[torch.empty_like(h, device=dev) for h in host] for _ in range(2)]
  ready = [torch.cuda.Event(), torch.cuda.Event()]
  consumed = [torch.cuda.Event(), torch.cuda.Event()]
  loss_slots = torch.zeros(2, dtype=torch.float32).pin_memory()
  loss_done = [torch.cuda.Event(), torch.cuda.Event()]
  losses_read = []

  def upload(i):
    slot = i & 1
    with torch.cuda.stream(copy_stream):
      copy_stream.wait_event(consumed[slot])       # add_batch of step i-2 has read this slot
      for d, h in zip(staged[slot], host):
        d.copy_(h, non_blocking=True)
      ready[slot].record(copy_stream)

  def e2e_step(i, last, read_prev=True):
    slot = i & 1
    main_stream.wait_event(ready[slot])
    if not last:
      upload(i + 1)
    d = staged[slot]
    if e2e_fns is not None:
      # add_batch + get_next + train of this staging slot replayed as ONE graph (one launch)
      out = e2e_fns[slot]()
      consumed[slot].record(main_stream)
    else:
      rb.add_batch(trajectory.Trajectory(d[0], d[1], d[2], (), d[3], d[4], d[5]))
      consumed[slot].record(main_stream)
      # get_next + train through common.function (the reference idiom: examples wrap
      # agent.train in common.function), i.e. the same captured step as `value`
      out = fn()[0].loss
    loss_slots[slot:slot + 1].copy_(out.reshape(1), non_blocking=True)   # device -> pinned host
    loss_done[slot].record(main_stream)
    if read_prev:                                  # read the PREVIOUS step's loss while this one runs
      loss_done[slot ^ 1].synchronize()
      losses_read.append(float(loss_slots[slot ^ 1]))

  def _fused(slot):
    d = staged[slot]

    def f():
      if not prefetch:
        rb.add_batch(trajectory.Trajectory(d[0], d[1], d[2], (), d[3], d[4], d[5]))
        exp_, _ = rb.get_next(sample_batch_size=B, num_steps=T)
        return agent.train(exp_).loss
      # collect-side work of this step (store the uploaded frames, draw the next batch) beside
      # the update on the batch drawn one step earlier
      main = torch.cuda.current_stream()
      side_stream.wait_stream(main)
      with torch.cuda.stream(side_stream):
        rb.add_batch(trajectory.Trajectory(d[0], d[1], d[2], (), d[3], d[4], d[5]))
        rb.get_next(sample_batch_size=B, num_steps=T, out=sample_bufs[slot ^ 1])
      loss_ = agent.train(sample_bufs[slot][0]).loss
      main.wait_stream(side_stream)
      return loss_
    return common.function(f, warmup=1)

  e2e_fns = [_fused(0), _fused(1)] if (use_graph and world == 1) else None
  for s in range(2):
    consumed[s].record(main_stream)
  upload(0)
  n_pre = 5 if e2e_fns is not None else 3          # both slot graphs: eager call + capture each
  for i in range(n_pre):
    e2e_step(i, False, read_prev=i > 0)
  sync_all()
  losses_read.clear()
  ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ee0.record()
  for i in range(Ke):                              # the first timed step has no timed predecessor
    e2e_step(n_pre + i, i == Ke - 1, read_prev=i > 0)
  loss_done[(n_pre + Ke - 1) & 1].synchronize()    # the last step's loss is read inside the region
  losses_read.append(float(loss_slots[(n_pre + Ke - 1) & 1]))
  ee1.record()
  sync_all()
  e2e_ms = ee0.elapsed_time(ee1)
  if world > 1:
    t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
  e2e_value = Ke / (e2e_ms / 1000.0) * world
  assert len(losses_read) == Ke and all(np.isfinite(losses_read)), 'e2e loss read-back incomplete'

  line = None
  if rank == 0:
    line = dict(
        metric='train steps/sec (DQN Atari-shape, batch 256)', value=value, unit='steps/s',
        n_gpus=world, steps=K, warmup=W, repeats=R, ms_per_step=ms / K,
        block_ms=[round(b, 4) for b in block_ms], higher_is_better=True,
        scaling='weak', vs_baseline=None, dtype='f32 (3xTF32 tensor-core GEMMs, fp32 accumulate)', data='synthetic',
        config=dict(workload=WORKLOAD, global_batch=B * world, per_gpu_batch=B, num_actions=A,
                    parallelism=f'dp{world}' if world > 1 else 'single',
                    multi_gpu=(None if world == 1 else
                               f'gradient all-reduce in buckets of {agent._bucket_bytes} B on a side '
                               f'stream beside the backward pass, dynamic GEMM tile scheduler, '
                               f'NCCL_MAX_CTAS={os.environ.get("NCCL_MAX_CTAS")}'),
                    l2='inputs > L2: 29.6 GB ring, fresh random rows every step',
                    cuda_graph=bool(use_graph), collect_frames_per_e2e_step=B_ENV,
                    input_pipeline=('prefetch(1): sample of step i+1 on a side stream beside train(i), two '
                                    'sample buffers' if prefetch else 'sample then train on one stream'),
                    timing=f'median of {R} blocks of {K} graph replays, each block bracketed by '
                           'barrier + synchronize, CUDA events, max over ranks',
                    e2e_pipeline='pinned host frames -> double-buffered H2D on a copy stream -> '
                                 'common.function(add_batch + get_next + train) per staging slot -> per-step loss '
                                 'D2H into pinned slots, read one step behind'),
        clocks=clk,
        e2e=dict(value=e2e_value, unit='steps/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=4,
                 steps=Ke, losses_read=len(losses_read)),
        gpu_launches=int(launches_per_step * K),
        roofline=dict(kernel='tc2_gemm_kernel / tc_gemm_kernel (Q-net conv/dense fwd+bwd, tcgen05 kind::tf32, 3xTF32)', bound='tensor',
                      achieved=update_tfs, peak=peaks['tensor'], unit='TFLOP/s',
                      frac=update_tfs / peaks['tensor'], traffic=traffic.get('update'),
                      peak_source=peaks['src'] + ' bf16 sustained', ms=update_ms,
                      algorithmic_flops=FLOPS_PER_STEP,
                      # fp32-equivalent ceiling of the arithmetic actually used: TF32 runs at half
                      # the bf16 rate and 3xTF32 issues three MMAs per product -> peak / 6
                      tf32x3_equiv_peak=peaks['tensor'] / 6.0,
                      frac_of_tf32x3_equiv=update_tfs / (peaks['tensor'] / 6.0)),
        roofline_gather=dict(kernel='row_copy_tma<MODE_SAMPLE> (cp.async.bulk)', bound='hbm', achieved=gather_gbs,
                             peak=peaks['hbm'], unit='GB/s', frac=gather_gbs / peaks['hbm'],
                             traffic=traffic.get('gather'), peak_source=peaks['src'],
                             us=gather_ms * 1e3, algorithmic_bytes=GATHER_BYTES),
        final_loss=final_loss)
    if parity is not None:
      line['parity'] = parity

  # The main measurement is complete: everything below (configs 1 / 3 / 4 / 5, the CPU arm) only
  # ADDS keys to the line.  A watchdog makes sure the line is printed even if one of them hangs
  # (e.g. a rank lost inside a collective at an untested world size): on expiry rank 0 prints what
  # it has and every rank leaves.
  import threading
  printed = threading.Lock()

  def emit(note=None):
    if not printed.acquire(blocking=False):
      return
    if rank == 0:
      out = dict(line)
      out.update(extra)
      if note:
        out['extras_note'] = note
      print(json.dumps(out), flush=True)

  def on_timeout():
    sys.stderr.write(f'[rank {rank}] extras exceeded {args.extras_timeout} s; printing the line without them\n')
    emit(f'watchdog: extras did not finish within {args.extras_timeout} s')
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)

  watchdog = threading.Timer(args.extras_timeout + (0 if rank == 0 else 5), on_timeout)
  watchdog.daemon = True
  watchdog.start()

  # ---- the other BASELINE configs (ring freed first: config 5 needs the HBM) --------------------
  del rb, st_store, obs_store, act_store, nst_store, rew_store, disc_store, exp, staged, train_only, e2e_fns
  del sample_bufs, bodies
  if use_graph:
    del fn
    if prefetch:
      del graphs
  torch.cuda.empty_cache()
  if not args.no_extra:
    from profiles import configs
    guarded('gather_sweep', lambda: configs.gather_sweep(
        dev, world, rank, peaks, caps_m=(1, 2, 4) if world == 1 else ((1, 4, 8) if world == 2 else (1, 4, 8, 16))))
    guarded('ppo_update', lambda: configs.ppo_update(strategy, dev, peaks))
    guarded('sac_step', lambda: configs.sac_step(strategy, dev, peaks))
    if world == 1:
      guarded('cartpole_iter', lambda: configs.cartpole_iter(dev))

  cpu = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    arm = CpuArm()
    sps, sweep, sample = arm.measure(8, 3)
    cpu = dict(value=sps, unit='steps/s', cores=arm.threads, kind='port', sample=sample,
               other_thread_counts=sweep, logical_cpus=os.cpu_count())

  if cpu is not None and line is not None:
    line['cpu_baseline'] = cpu
  watchdog.cancel()
  emit()
  if world > 1:
    # CUDA graphs that captured NCCL kernels make the communicator teardown hang on this stack:
    # leave without running destructors once every rank is done (or after a minute, if a rank
    # never arrives).
    leave = threading.Timer(60.0, lambda: os._exit(0))
    leave.daemon = True
    leave.start()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == '__main__':
  main()
