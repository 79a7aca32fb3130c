"""ctypes binding of libb200rl.so (include/b200rl.h).

The product path has NO CPU fallback: if the shared library is missing or the device is not a
CUDA device, calls raise.  `lib()` loads lazily so that host-only logic (specs, nests, shape
validation) stays importable on a CPU-only box.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200RL_LIB: an alternative build of the same library (profiles/ A/B runs of compile-time variants)
LIB_PATH = os.environ.get('B200RL_LIB') or os.path.join(_HERE, 'lib', 'libb200rl.so')

MAX_LEAVES = 24
ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2
LOSS_HUBER, LOSS_SQUARED = 0, 1

c_void_p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_u64 = ctypes.c_uint64
c_int = ctypes.c_int
c_f32 = ctypes.c_float
c_f64 = ctypes.c_double


class Leaf(ctypes.Structure):
  _fields_ = [('storage', c_void_p), ('row_bytes', c_i64)]


class Ring(ctypes.Structure):
  _fields_ = [
      ('num_leaves', ctypes.c_int32),
      ('_pad', ctypes.c_int32),
      ('batch_size', c_i64),
      ('max_length', c_i64),
      ('id_table', c_void_p),
      ('last_id', c_void_p),
      ('ticket', c_void_p),
      ('leaves', Leaf * MAX_LEAVES),
  ]


class ConvGeom(ctypes.Structure):
  _fields_ = [(n, ctypes.c_int32) for n in ('N', 'H', 'W', 'C', 'KH', 'KW', 'F', 'stride')
             ] + [('x_batch_stride', ctypes.c_int64)]


class PpoKl(ctypes.Structure):
  _fields_ = [('old_loc', c_void_p), ('old_scale', c_void_p), ('ld_old', c_i64),
              ('terms', c_void_p), ('grad_scale', c_f32)]


class B200RLError(RuntimeError):
  pass


# name -> argtypes (restype is int unless listed in _RESTYPES)
_P = c_void_p
SIGNATURES = {
    'b200rl_set_copy_variant': [c_int],
    'b200rl_set_pdl': [c_int],
    'b200rl_rb_add_batch': [ctypes.POINTER(Ring), _P, _P],
    'b200rl_rb_sample': [ctypes.POINTER(Ring), c_i64, c_i64, _P, _P, c_u64, _P, _P, _P, _P, _P,
                         _P, _P],
    'b200rl_rb_read_rows': [ctypes.POINTER(Ring), _P, c_i64, _P, _P, _P],
    'b200rl_rb_write_rows': [ctypes.POINTER(Ring), _P, c_i64, _P, _P],
    'b200rl_rb_gather_all': [ctypes.POINTER(Ring), c_i64, _P, _P],
    'b200rl_rb_clear': [ctypes.POINTER(Ring), c_int, _P],
    'b200rl_ep_assign': [_P, _P, _P, _P, _P, c_i64, c_i64, c_i64, c_i64, _P, _P, _P, _P, _P, c_int, c_int,
                         _P, _P, _P],
    'b200rl_rb_draw': [ctypes.POINTER(Ring), c_i64, c_i64, c_u64, _P, _P, _P, _P],
    'b200rl_discounted_return': [_P, _P, _P, _P, c_i64, c_i64, c_int, c_int, _P],
    'b200rl_gae': [_P, _P, _P, _P, c_f32, _P, c_i64, c_i64, c_int, _P],
    'b200rl_discounted_return_ld': [_P, _P, _P, _P, c_i64, c_i64, c_i64, c_i64, c_i64, _P],
    'b200rl_gae_ld': [_P, _P, _P, _P, c_f32, _P, c_i64, c_i64, c_i64, c_i64, c_i64, _P],
    'b200rl_ppo_loss': [_P, _P, c_i64, _P, _P, _P, _P, _P, _P, _P, c_i64, c_i64, c_i64, c_f32, c_f32,
                        c_f32, c_f32, c_f32, c_f32, _P, _P, _P, c_i64, _P, _P, _P, _P, c_i64, _P],
    'b200rl_ppo_kl': [_P, _P, c_i64, _P, _P, c_i64, _P, c_i64, c_i64, c_f32, _P, _P, _P, c_i64, _P],
    'b200rl_ppo_kl_terms': [_P, _P, c_f32, c_f32, c_f32, _P, _P],
    'b200rl_ppo_kl_beta_update': [_P, _P, c_f32, c_f32, _P],
    'b200rl_normal_logp': [_P, _P, c_i64, _P, c_i64, c_i64, _P, _P],
    'b200rl_normal_sample': [_P, _P, c_i64, c_i64, c_i64, _P, _P, c_u64, _P, _P, _P],
    'b200rl_normal_proj_fwd': [_P, _P, _P, _P, c_i64, c_i64, _P, _P, _P],
    'b200rl_normal_proj_bwd': [_P, _P, _P, _P, _P, _P, c_i64, c_i64, _P, _P, _P],
    'b200rl_colsum': [_P, _P, c_int, c_i64, c_i64, c_f32, _P, _P, c_i64, _P],
    'b200rl_normalize': [_P, _P, c_i64, c_i64, _P, _P, _P, c_f32, c_f32, _P],
    'b200rl_normalizer_update': [_P, _P, _P, _P, _P, _P, c_f32, c_i64, _P],
    'b200rl_ppo_discounts': [_P, _P, c_f32, c_i64, _P, _P],
    'b200rl_ppo_weights': [_P, _P, _P, _P, c_i64, _P, _P],
    'b200rl_sac_sample': [_P, c_i64, c_i64, _P, _P, _P, c_u64, _P, _P, c_i64, _P, _P, _P, _P],
    'b200rl_sac_sample_bwd': [_P, _P, _P, _P, _P, _P, _P, c_i64, _P, c_i64, c_i64, _P, _P],
    'b200rl_sac_critic_loss': [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_i64, c_f32, c_f32, c_f32,
                               c_f32, _P, _P, _P, _P, _P, _P],
    'b200rl_sac_actor_loss': [_P, _P, _P, _P, _P, c_i64, c_f32, c_f32, _P, _P, _P, _P, _P, _P],
    'b200rl_sac_alpha_loss': [_P, _P, _P, c_i64, c_f32, c_int, c_f32, c_f32, _P, _P, _P, _P],
    'b200rl_concat2': [_P, c_i64, c_i64, _P, c_i64, c_i64, c_i64, _P, _P],
    'b200rl_nstep_reduce': [_P, _P, c_f64, _P, _P, c_i64, c_i64, _P],
    'b200rl_dqn_td_loss': [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_i64, c_i64, c_i64, c_i64, c_i64,
                           c_f64, c_f64, c_int, c_f32, _P, _P, _P, _P, _P, _P],
    'b200rl_set_gemm_mode': [c_int],
    'b200rl_set_tc2_flags': [c_int],
    'b200rl_set_tile_scheduler': [c_int],
    'b200rl_tc2_trace_buffer': [_P],
    'b200rl_dense_fwd': [_P, c_i64, _P, _P, _P, c_i64, c_i64, c_i64, c_int, _P, c_i64, _P],
    'b200rl_dense_fwd_pair': [_P, _P, c_i64, _P, _P, _P, _P, _P, _P, c_i64, c_i64, c_i64, c_int, _P,
                              c_i64, _P],
    'b200rl_conv2d_fwd_pair': [_P, _P, c_int, c_f32, _P, _P, _P, _P, _P, _P,
                               ctypes.POINTER(ConvGeom), c_int, _P, c_i64, _P],
    'b200rl_dense_bwd': [_P, c_i64, _P, _P, _P, _P, _P, c_i64, c_i64, c_i64, c_int, c_int, _P, c_i64,
                         _P],
    'b200rl_act_bwd': [_P, _P, _P, c_i64, c_int, _P],
    'b200rl_conv2d_fwd': [_P, c_int, c_f32, _P, _P, _P, ctypes.POINTER(ConvGeom), c_int, _P,
                          c_i64, _P],
    'b200rl_conv2d_bwd': [_P, c_int, c_f32, _P, _P, _P, _P, _P, ctypes.POINTER(ConvGeom), c_int,
                          c_int, _P, c_i64, _P],
    'b200rl_adam_tf': [_P, _P, _P, _P, c_i64, c_f32, c_f32, c_f32, c_f32, _P, _P, _P],
    'b200rl_rmsprop_tf': [_P, _P, _P, _P, _P, c_i64, c_f32, c_f32, c_f32, c_f32, c_int, _P, _P],
    'b200rl_soft_update': [_P, _P, c_i64, c_f32, c_i64, _P, _P],
    'b200rl_clip_by_norm_segments': [_P, _P, c_i64, c_f32, _P],
    'b200rl_global_norm_scale': [_P, c_i64, c_f32, _P, _P, _P, c_i64, _P],
    'b200rl_add_scaled': [_P, _P, c_i64, c_f32, _P],
    'b200rl_l2_sum': [_P, c_i64, c_f32, _P, _P],
    'b200rl_counter_add': [_P, c_i64, _P],
    'b200rl_shuffle_order': [c_i64, c_i64, c_u64, c_u64, _P],
    'b200rl_rb_gather_frame_stack': [_P, _P, c_i64, c_i64, _P, _P, c_i64, c_i64, c_int, _P, _P],
    'b200rl_epsilon_greedy': [_P, _P, c_i64, c_i64, c_f32, c_u64, _P, _P, _P, _P, _P],
    'b200rl_env_random_step': [_P, _P, _P, c_i64, c_int, _P, _P, c_i64, c_f32, c_u64, _P, _P],
    'b200rl_env_cartpole_step': [_P, _P, _P, _P, _P, _P, _P, c_i64, ctypes.c_int32, c_u64, _P,
                                 _P],
}
_RESTYPES = {
    'b200rl_last_error': ctypes.c_char_p,
    'b200rl_version': c_int,
    'b200rl_launch_count': c_i64,
    'b200rl_get_pdl': c_int,
}

_lib = None


def lib():
  """Returns the loaded CDLL; raises if libb200rl.so has not been built."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise B200RLError(
          f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
          '(or agents_b200/csrc/build.sh). There is no CPU fallback for the hot path.')
    l = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
      fn = getattr(l, name)
      fn.argtypes = argtypes
      fn.restype = c_int
    for name, res in _RESTYPES.items():
      fn = getattr(l, name)
      fn.argtypes = []
      fn.restype = res
    _lib = l
  return _lib


def call(name, *args):
  """Calls an int-returning entry point and raises B200RLError on a non-zero status."""
  l = lib()
  rc = getattr(l, name)(*args)
  if rc != 0:
    msg = l.b200rl_last_error().decode('utf-8', 'replace')
    if rc == -1:
      raise ValueError(msg)
    raise B200RLError(f'{name} failed ({rc}): {msg}')
  return rc


def launch_count():
  return int(lib().b200rl_launch_count())


def ptr(t):
  """Device pointer of a torch tensor (None -> NULL). Requires a CUDA, contiguous tensor."""
  if t is None:
    return None
  if not t.is_cuda:
    raise B200RLError('libb200rl needs CUDA tensors: there is no CPU fallback '
                      f'(got a tensor on {t.device}).')
  if not t.is_contiguous():
    raise B200RLError('libb200rl needs contiguous tensors.')
  return t.data_ptr()


def dptr(t):
  """Device pointer of a possibly batch-strided CUDA tensor (stride handled by the callee)."""
  if not t.is_cuda:
    raise B200RLError('libb200rl needs CUDA tensors: there is no CPU fallback '
                      f'(got a tensor on {t.device}).')
  return t.data_ptr()


def stream():
  import torch
  return torch.cuda.current_stream().cuda_stream


def ptr_array(tensors):
  """Host array of device pointers (kept alive by the caller for the duration of the call)."""
  arr = (c_void_p * len(tensors))()
  for i, t in enumerate(tensors):
    arr[i] = ptr(t)
  return arr
