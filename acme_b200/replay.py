"""Reverb-shaped replay facade over the GPU-resident replay shard (libb200rl).

Mirrors the client surface the reference's hot path uses (SURVEY.md §8b):
  reverb.Table / selectors / rate_limiters / Server      acme/agents/tf/dqn/agent.py:95-102
  reverb.Client.writer / Writer.create_item / close      acme/adders/reverb/base.py:111-132,
                                                         acme/adders/reverb/transition.py:162-165
  reverb.TFClient.update_priorities                      acme/agents/tf/dqn/learning.py:151-154
  reverb.Client.mutate_priorities                        acme/agents/jax/dqn/learning.py:131-134
  reverb.ReplaySample / SampleInfo dtypes                acme/testing/fakes.py:245-262
  datasets.make_reverb_dataset                           acme/datasets/reverb.py:36-139

Everything that touches data (ring writes, sampling, gather, n-step build, priority updates)
runs in CUDA through the C ABI; this module only keeps handles and packs nests into byte rows.
"""

from __future__ import annotations

import ctypes as C
import itertools
import threading
from typing import Any, Dict, List, NamedTuple, Optional, Sequence

import numpy as np

from acme_b200 import _capi, tree

DEFAULT_PRIORITY_TABLE = 'priority_table'  # acme/adders/reverb/base.py:30


class SampleInfo(NamedTuple):
  key: Any           # uint64 [B]
  probability: Any   # float64 [B]
  table_size: Any    # int64 [B]
  priority: Any      # float64 [B]


class ReplaySample(NamedTuple):
  info: SampleInfo
  data: Any


# ----------------------------------------------------------------------------- table configuration
class selectors:  # namespace, like reverb.selectors

  class Prioritized:

    def __init__(self, priority_exponent: float):
      self.priority_exponent = float(priority_exponent)

  class Uniform:
    priority_exponent = 0.0  # P(i) = w_i^0 / sum = 1/N

  class Fifo:
    pass


class rate_limiters:  # namespace, like reverb.rate_limiters

  class MinSize:

    def __init__(self, min_size_to_sample: int):
      self.min_size_to_sample = int(min_size_to_sample)


class _Packer:
  """Packs a nest of arrays (per a nest of specs) into one contiguous byte row and back."""

  def __init__(self, spec_nest):
    self.structure = spec_nest
    self.leaves = []
    off, row_align = 0, 1
    for s in tree.flatten(spec_nest):
      dt = np.dtype(s.dtype)
      shape = tuple(int(d) for d in s.shape)
      n = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
      align = min(dt.itemsize, 16)
      row_align = max(row_align, align)
      off = -(-off // align) * align
      self.leaves.append((shape, dt, off, n))
      off += n
    # rows of a batch are `nbytes` apart: the row size must keep EVERY leaf aligned in rows b > 0 too
    # (a {float32[3], uint8[1]} nest is 13 bytes of payload in a 16-byte row)
    self.nbytes = -(-off // row_align) * row_align
    self.single = len(self.leaves) == 1 and not tree.is_nest(spec_nest)

  def pack(self, value_nest) -> np.ndarray:
    if self.single:
      # one leaf (the usual observation / action): hand the array's own bytes to the C layer, which copies them into
      # pinned staging during the call -- no intermediate row
      shape, dt, _, n = self.leaves[0]
      a = np.asarray(value_nest, dtype=dt)
      if a.shape != shape:
        raise ValueError(f'expected shape {shape}, got {a.shape}')
      if n and a.flags.c_contiguous:
        return a.reshape(-1).view(np.uint8)
    row = np.zeros(max(self.nbytes, 1), np.uint8)
    vals = tree.flatten(value_nest)
    if len(vals) != len(self.leaves):
      raise ValueError('value does not match the table signature')
    for v, (shape, dt, off, n) in zip(vals, self.leaves):
      a = np.asarray(v, dtype=dt)
      if a.shape != shape:
        raise ValueError(f'expected shape {shape}, got {a.shape}')
      row[off:off + n] = np.frombuffer(a.tobytes(), np.uint8)
    return row

  def unpack_batch(self, rows):
    """rows: torch uint8 [..., nbytes] -> nest of torch tensors [..., *shape] (views)."""
    import torch
    out = []
    lead = tuple(rows.shape[:-1])
    for shape, dt, off, n in self.leaves:
      tdt = getattr(torch, dt.name) if dt.name != 'bool' else torch.bool
      out.append(rows[..., off:off + n].view(tdt).reshape(lead + shape) if n else
                 torch.empty(lead + shape, dtype=tdt, device=rows.device))
    return tree.unflatten_as(self.structure, out)


class Table:
  """reverb.Table: configuration + (once placed on a device) the GPU replay shard."""

  def __init__(self, name: str, sampler, remover, max_size: int, rate_limiter, signature=None,
               slot_capacity: Optional[int] = None, max_window: int = 8, discount: float = 0.99,
               device: int = 0, shard_count: int = 1, shard_rank: int = 0, stage_slots: int = 0, frame_stack: int = 0):
    """frame_stack = F > 1 (SURVEY §8f-1): the observation is a uint8 stack of F frames on its LAST axis, as
    `FrameStacker` / `AtariWrapper` produce it (`acme/wrappers/frame_stacking.py:64-88`, `atari_wrapper.py:277-308`: the
    newest frame last, blank frames before the episode's first observation).  The last axis may also hold C * F bytes:
    the stack of F frames of C channels ([..., C, F]) flattened, as `AtariWrapper(grayscaling=False)` gives it; its byte
    c * F + f is channel c of frame f (f = F - 1 the newest), the bytes of [..., C, F] in the same order, so both
    layouts are one ring layout.  The HBM ring then stores ONE frame per
    step and K3 rebuilds the stacks when it gathers: obs_bytes / F bytes per step (7,056 instead of 28,224 for Atari)
    and F times less host-to-device traffic per insert.  The caller's observations must really be such stacks: the
    older F-1 frames of every observation are taken from the previous observations of the same episode."""
    if not isinstance(remover, selectors.Fifo):
      raise NotImplementedError('only the Fifo remover is implemented (the one the hot path uses)')
    self.name = name
    self.alpha = float(getattr(sampler, 'priority_exponent'))
    self.max_size = int(max_size)
    self.min_size = int(getattr(rate_limiter, 'min_size_to_sample', 1))
    self.signature = signature
    self.max_window = int(max_window)
    self.discount = np.float32(discount)
    self.device = device
    self.shard_count, self.shard_rank = shard_count, shard_rank
    self.stage_slots = stage_slots
    self.frame_stack = int(frame_stack) if frame_stack and frame_stack > 1 else 0
    # one slot per observation; an episode of T steps uses T+1 slots and yields >= T items, so
    # 2*max_size (+window) slots can never evict a live item before the Fifo remover does.
    self.slot_capacity = int(slot_capacity) if slot_capacity else 2 * self.max_size + self.max_window + 2 + self.frame_stack
    self._handle = None
    self._lock = threading.Lock()
    self.is_sequence = False
    if signature is not None:
      self._bind(signature)

  @classmethod
  def priorities_only(cls, name: str, priority_exponent: float, max_size: int, device: int = 0,
                      shard_count: int = 1, shard_rank: int = 0) -> 'Table':
    """A table that holds only the sum tree (no payload ring): sampling / update sweeps."""
    t = cls(name, selectors.Prioritized(priority_exponent), selectors.Fifo(), max_size,
            rate_limiters.MinSize(1), signature=None, device=device, shard_count=shard_count,
            shard_rank=shard_rank)
    t.signature = ()
    t.obs_packer = t.act_packer = _Packer(())
    t.has_extras = False
    t.is_sequence = False
    return t

  # -- lifecycle
  def _bind(self, signature):
    # a `Step` of specs (adders.SequenceAdder.signature): items are sequences of whole steps (SURVEY §8f-3); the row
    # stored beside each observation is (action, start_of_episode, extras)
    self.is_sequence = 'start_of_episode' in getattr(signature, '_fields', ())
    if self.is_sequence:
      self.obs_packer = _Packer(signature.observation)
      self.act_packer = _Packer((signature.action, signature.start_of_episode, signature.extras))
      self.has_extras = True
      self.signature = signature
      if self.frame_stack:
        raise ValueError('frame_stack is not supported for sequence tables')
      return
    sig = tuple(signature)
    extras_spec = sig[5] if len(sig) > 5 else ()
    self.obs_packer = _Packer(sig[0])
    self.act_packer = _Packer((sig[1], extras_spec) if extras_spec != () else sig[1])
    self.has_extras = extras_spec != ()
    self.signature = sig
    if self.frame_stack:
      leaves = tree.flatten(sig[0])
      shape = tuple(leaves[0].shape) if len(leaves) == 1 else ()
      if len(leaves) != 1 or np.dtype(leaves[0].dtype) != np.uint8 or not shape or shape[-1] % self.frame_stack != 0:
        raise ValueError(f'frame_stack={self.frame_stack} needs a single uint8 observation whose last axis is the frame stack '
                         f'([..., F]) or C channels of F frames flattened ([..., C * F]); got {sig[0]}')

  def _ensure(self):
    if self._handle is not None:
      return
    with self._lock:      # actor threads and the learner thread may all touch a fresh table first (ctypes drops the GIL)
      self._ensure_locked()

  def _ensure_locked(self):
    if self._handle is not None:
      return
    if self.signature is None:
      raise ValueError(f'table {self.name!r} has no signature; pass signature=Adder.signature(spec)')
    _capi.require_device(self.device)
    cfg = _capi.ReplayCfg(max_items=self.max_size, slot_capacity=self.slot_capacity,
                          obs_bytes=self.obs_packer.nbytes, act_bytes=self.act_packer.nbytes,
                          max_window=self.max_window, shard_count=self.shard_count,
                          shard_rank=self.shard_rank, device=self.device,
                          stage_slots=self.stage_slots, frame_stack=self.frame_stack, gamma=float(self.discount),
                          alpha=self.alpha)
    h = C.c_void_p()
    _capi.call('b200rl_replay_create', C.byref(h), C.byref(cfg))
    self._handle = h

  @property
  def handle(self):
    self._ensure()
    return self._handle

  def close(self):
    if self._handle is not None:
      _capi.load().b200rl_replay_destroy(self._handle)
      self._handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:  # noqa: BLE001
      pass

  # -- host view
  def info(self):
    size, head, tail, mass = C.c_int64(), C.c_uint64(), C.c_uint64(), C.c_float()
    _capi.call('b200rl_replay_info', self.handle, C.byref(size), C.byref(head), C.byref(tail),
               C.byref(mass), _capi.current_stream())
    return dict(size=size.value, head_key=head.value, tail_key=tail.value, total_mass=mass.value)

  @property
  def size(self) -> int:
    size = C.c_int64()
    _capi.call('b200rl_replay_info', self.handle, C.byref(size), None, None, None, None)
    return size.value

  def can_sample(self, batch_size: int = 1) -> bool:
    return self.size >= max(self.min_size, 1)

  def flush(self):
    _capi.call('b200rl_replay_flush', self.handle, _capi.current_stream())

  def reset(self):
    _capi.call('b200rl_replay_reset', self.handle, _capi.current_stream())

  def open_writer(self) -> int:
    """A new writer id on this table (`b200rl_writer_open`), for append_multi."""
    w = C.c_int32()
    _capi.call('b200rl_writer_open', self.handle, C.byref(w))
    return w.value

  def append_multi(self, writers, obs, act, reward, discount, first, last, n_step: int, priority: float = 1.0):
    """One step of many episodes in one insert (`b200rl_writer_append_multi`): element i is the next timestep of writer
    writers[i], with NStepTransitionAdder's items over `n_step` and raw priority `priority`.  obs: [n, *obs_shape] -- a
    CUDA tensor is read on the device, anything else as host rows; act [n, *action_shape] (host), the action taken from
    obs[i] (ignored where last[i]); reward / discount [n], what followed it; first / last [n] bools.  Only transition
    tables without extras whose observation and action are single arrays."""
    if self.is_sequence or self.has_extras or not (self.obs_packer.single and self.act_packer.single):
      raise ValueError(f'table {self.name!r}: append_multi writes transition tables without extras whose observation '
                       'and action are single arrays')
    writers = np.ascontiguousarray(writers, np.int32)
    n = writers.size
    on_device = bool(getattr(obs, 'is_cuda', False))
    if on_device:
      if not obs.is_contiguous() or obs.numel() * obs.element_size() != n * self.obs_packer.nbytes:
        raise ValueError(f'obs must be {n} contiguous rows of {self.obs_packer.nbytes} bytes')
    else:
      obs = np.ascontiguousarray(obs, self.obs_packer.leaves[0][1])
      if obs.nbytes != n * self.obs_packer.nbytes:
        raise ValueError(f'obs must be {n} rows of {self.obs_packer.nbytes} bytes')
    act = np.ascontiguousarray(act, self.act_packer.leaves[0][1])
    if act.nbytes != n * self.act_packer.nbytes:
      raise ValueError(f'act must be {n} rows of {self.act_packer.nbytes} bytes')
    rew = np.ascontiguousarray(reward, np.float32).reshape(n)
    disc = np.ascontiguousarray(discount, np.float32).reshape(n)
    first = np.ascontiguousarray(first, np.uint8).reshape(n)
    last = np.ascontiguousarray(last, np.uint8).reshape(n)
    _capi.call('b200rl_writer_append_multi', self.handle, n, writers.ctypes.data, _capi.ptr(obs), int(on_device),
               act.ctypes.data, rew.ctypes.data, disc.ctypes.data, first.ctypes.data, last.ctypes.data, int(n_step),
               float(priority), _capi.current_stream())

  def tree_levels(self):
    L, F, S = C.c_int32(), C.c_int32(), C.c_int32()
    _capi.call('b200rl_replay_tree_levels', self.handle, C.byref(L), C.byref(F), C.byref(S))
    return L.value, F.value, S.value

  def read_tree_level(self, level: int) -> np.ndarray:
    w = C.c_int64()
    _capi.call('b200rl_replay_tree_level_width', self.handle, level, C.byref(w))
    out = np.empty(w.value, np.float32)
    _capi.call('b200rl_replay_tree_read', self.handle, level, out.ctypes.data, w.value,
               _capi.current_stream())
    return out

  def read_tree_prefix(self, level: int) -> np.ndarray:
    w = C.c_int64()
    _capi.call('b200rl_replay_tree_level_width', self.handle, level, C.byref(w))
    out = np.empty(w.value, np.float32)
    _capi.call('b200rl_replay_tree_read_prefix', self.handle, level, out.ctypes.data, w.value,
               _capi.current_stream())
    return out

  def mass_ptr(self) -> int:
    p = C.c_void_p()
    _capi.call('b200rl_replay_mass_ptr', self.handle, C.byref(p))
    return p.value

  def mass_tensor(self):
    """The shard's total mass M_r as a zero-copy device tensor [1] (the tree's root)."""
    import torch
    return torch.as_tensor(_MassView(self.mass_ptr()), device=torch.device('cuda', self.device))

  def set_global_mass(self, total):
    """Installs sum_r M_r (device float tensor [1], kept alive by the table) so that K1 reports weight / sum_r M_r
    (global-priority-mass normalisation, SURVEY §8e); None restores weight / (R * M_r)."""
    self._global_mass = total
    _capi.call('b200rl_replay_set_global_mass', self.handle, None if total is None else total.data_ptr())

  # -- device path (torch tensors are only memory handles here)
  def sample_into(self, u, idx, keys, prob, stratified=True):
    _capi.call('b200rl_replay_sample', self.handle, u.shape[0], _capi.ptr(u), int(stratified),
               _capi.ptr(idx), _capi.ptr(keys), _capi.ptr(prob), _capi.current_stream())

  def gather_into(self, idx, o_tm1, a_tm1, R, D, o_t):
    _capi.call('b200rl_replay_gather', self.handle, idx.shape[0], _capi.ptr(idx), _capi.ptr(o_tm1),
               _capi.ptr(a_tm1), _capi.ptr(R), _capi.ptr(D), _capi.ptr(o_t), _capi.current_stream())

  def gather_rows_into(self, idx, o_tm1, a_tm1, R, D, o_t, rows_tm1_ptr: int, rows_t_ptr: int, geom):
    """K3 that also writes the first conv layer's bf16 row images (`b200rl_replay_gather_rows`)."""
    _capi.call('b200rl_replay_gather_rows', self.handle, idx.shape[0], _capi.ptr(idx), _capi.ptr(o_tm1), _capi.ptr(a_tm1),
               _capi.ptr(R), _capi.ptr(D), _capi.ptr(o_t), rows_tm1_ptr, rows_t_ptr, geom, _capi.current_stream())

  def update_priorities_device(self, keys, priorities):
    _capi.call('b200rl_replay_update_priorities', self.handle, keys.shape[0], _capi.ptr(keys),
               _capi.ptr(priorities), _capi.current_stream())

  # -- core.Saveable: the whole shard (SURVEY §8f-4).  The reference's checkpointers save learner state only
  # (`acme/tf/savers.py:76-167`); a table restored here continues exactly where the saved one stopped: same keys, same
  # FIFO position, same priorities, open writers keep their episode windows.
  _SEGMENTS = ('obs', 'act', 'rew', 'disc', 'next', 'item_start', 'item_end', 'item_len', 'tree', 'key_range', 'item_prev')

  def _segment(self, which: int):
    import torch
    p, n = C.c_void_p(), C.c_int64()
    _capi.call('b200rl_replay_segment', self.handle, which, C.byref(p), C.byref(n))
    if not n.value:
      return None
    return torch.as_tensor(_RawBytes(p.value, n.value), device=torch.device('cuda', self.device))

  def save(self):
    """Host copy of the shard: {'host': bookkeeping blob, 'segments': {name: uint8 array}, 'geometry': ...}.  Staged
    steps are flushed first.  The observation ring is copied whole (28 KB per Atari slot): size the table accordingly."""
    import torch
    st = _capi.current_stream()
    size = C.c_int64()
    _capi.call('b200rl_replay_host_state', self.handle, None, 0, C.byref(size), st)
    blob = np.empty(size.value, np.uint8)
    _capi.call('b200rl_replay_host_state', self.handle, blob.ctypes.data, size.value, C.byref(size), st)
    torch.cuda.current_stream().synchronize()
    segs = {}
    for which, name in enumerate(self._SEGMENTS):
      t = self._segment(which)
      if t is not None:
        segs[name] = t.cpu().numpy()
    return dict(host=blob[:size.value].copy(), segments=segs,
                geometry=dict(max_size=self.max_size, slot_capacity=self.slot_capacity, alpha=self.alpha,
                              obs_bytes=self.obs_packer.nbytes, act_bytes=self.act_packer.nbytes,
                              frame_stack=self.frame_stack))

  def restore(self, state):
    import torch
    geo = state['geometry']
    if (geo['max_size'], geo['slot_capacity'], geo['obs_bytes'], geo['act_bytes'], geo.get('frame_stack', 0)) != (
        self.max_size, self.slot_capacity, self.obs_packer.nbytes, self.act_packer.nbytes, self.frame_stack):
      raise ValueError(f'table geometry differs from the saved one: {geo}')
    blob = np.ascontiguousarray(state['host'], np.uint8)
    _capi.call('b200rl_replay_set_host_state', self.handle, blob.ctypes.data, blob.size)
    for which, name in enumerate(self._SEGMENTS):
      t = self._segment(which)
      if t is not None:
        t.copy_(torch.as_tensor(np.ascontiguousarray(state['segments'][name], np.uint8)))
    torch.cuda.current_stream().synchronize()

  def set_weights(self, weights):
    """Priorities-only table (sampling/update sweeps): leaves <- weights (device f32 [n])."""
    _capi.call('b200rl_replay_set_weights', self.handle, weights.shape[0], _capi.ptr(weights),
               _capi.current_stream())


# ----------------------------------------------------------------------------- server / client
_SERVERS: Dict[int, 'Server'] = {}
_PORTS = itertools.count(41000)


class Server:
  """reverb.Server([tables], port=None): in-process registry of tables (no RPC: the data path is
  device memory, the 'address' only lets Client(...) find the tables like the reference does)."""

  def __init__(self, tables: Sequence[Table], port: Optional[int] = None):
    self.tables = {t.name: t for t in tables}
    self.port = port if port is not None else next(_PORTS)
    _SERVERS[self.port] = self

  def stop(self):
    _SERVERS.pop(self.port, None)
    for t in self.tables.values():
      t.close()

  def localhost_client(self) -> 'Client':
    return Client(f'localhost:{self.port}')


def _resolve(server_or_address) -> Server:
  if isinstance(server_or_address, Server):
    return server_or_address
  port = int(str(server_or_address).rsplit(':', 1)[-1])
  if port not in _SERVERS:
    raise ConnectionError(f'no acme_b200 replay server at {server_or_address!r}')
  return _SERVERS[port]


class Writer:
  """reverb.Writer re-cast for a ring of steps: append one environment step, then create items over
  the trailing `num_timesteps` steps (Reverb's own create_item meaning)."""

  def __init__(self, client: 'Client', max_sequence_length: int, delta_encoded=False, chunk_length=None):
    self._client = client
    self.max_sequence_length = max_sequence_length
    self._ids: Dict[str, int] = {}
    self._started = set()      # tables that already hold this episode's first observation
    self.closed = False

  def _wid(self, table: Table) -> int:
    if table.name not in self._ids:
      w = C.c_int32()
      _capi.call('b200rl_writer_open', table.handle, C.byref(w))
      self._ids[table.name] = w.value
    return self._ids[table.name]

  def append_step(self, observation, action, reward, discount, next_observation, extras=(),
                  tables: Optional[Sequence[str]] = None, start_of_episode: bool = False):
    if self.closed:
      raise RuntimeError('writer is closed')
    for name in (tables or self._client.server.tables):
      t = self._client.server.tables[name]
      # the ring stores every observation once: `observation` is only needed for the first step of an episode
      # (later it is the previous call's next_observation, already in the ring; the C layer ignores the pointer)
      obs = None if name in self._started else t.obs_packer.pack(observation)
      nxt = t.obs_packer.pack(next_observation)
      if getattr(t, 'is_sequence', False):
        act = t.act_packer.pack((action, np.bool_(start_of_episode), extras))
      else:
        act = t.act_packer.pack((action, extras) if t.has_extras else action)
      _capi.call('b200rl_writer_append', t.handle, self._wid(t), None if obs is None else obs.ctypes.data,
                 act.ctypes.data, float(np.float32(reward)), float(np.float32(discount)), nxt.ctypes.data)
      self._started.add(name)

  def create_item(self, table: str, num_timesteps: int, priority: float) -> int:
    if self.closed:
      raise RuntimeError('writer is closed')
    t = self._client.server.tables[table]
    key = C.c_uint64()
    _capi.call('b200rl_writer_create_item', t.handle, self._wid(t), int(num_timesteps),
               float(priority), C.byref(key))
    return key.value

  def close(self):
    if self.closed:
      raise RuntimeError('writer is already closed')
    for name, wid in self._ids.items():
      t = self._client.server.tables[name]
      if t._handle is not None:
        _capi.call('b200rl_writer_close', t.handle, wid)
    self.closed = True


class Client:
  """reverb.Client / reverb.TFClient in one object (same process, same device)."""

  def __init__(self, server_address):
    self.server = _resolve(server_address)
    self.server_address = f'localhost:{self.server.port}'

  def writer(self, max_sequence_length: int, delta_encoded: bool = False, chunk_length=None) -> Writer:
    return Writer(self, max_sequence_length, delta_encoded, chunk_length)

  def table(self, name: str) -> Table:
    return self.server.tables[name]

  def reset(self, table: str):
    self.server.tables[table].reset()

  # TFClient.update_priorities(table, keys, priorities)  (dqn/learning.py:153-154)
  def update_priorities(self, table: str, keys, priorities):
    import torch
    t = self.server.tables[table]
    if not (hasattr(keys, 'data_ptr') and keys.is_cuda):
      keys = torch.as_tensor(np.asarray(keys, np.uint64).view(np.int64)).cuda(t.device).view(torch.uint64)
    if not (hasattr(priorities, 'data_ptr') and priorities.is_cuda):
      priorities = torch.as_tensor(np.asarray(priorities, np.float64).astype(np.float32)).cuda(t.device)
    elif priorities.dtype != torch.float32:
      priorities = priorities.to(torch.float32)
    t.update_priorities_device(keys, priorities)

  # Client.mutate_priorities(table, updates={key: priority})  (jax/dqn/learning.py:133-134)
  def mutate_priorities(self, table: str, updates: Dict[int, float]):
    if updates:
      self.update_priorities(table, np.fromiter(updates.keys(), np.uint64, len(updates)),
                             np.fromiter(updates.values(), np.float64, len(updates)))


TFClient = Client


# ----------------------------------------------------------------------------- dataset
class _RawBytes:
  """A device byte range dressed up for torch.as_tensor (zero copy)."""

  def __init__(self, ptr: int, n: int):
    self.__cuda_array_interface__ = {'shape': (n,), 'typestr': '|u1', 'data': (ptr, False), 'version': 2}


class _MassView:
  """The tree's root mass (one device float) as a zero-copy array for torch.as_tensor."""

  def __init__(self, ptr: int):
    self.__cuda_array_interface__ = {'shape': (1,), 'typestr': '<f4', 'data': (ptr, False), 'version': 2}


class ReplayDataset:
  """What `make_reverb_dataset(...)` returns: an iterable of batched ReplaySamples living in HBM.

  Each `next()` = one K1 launch (sample) + one K3 launch (gather + n-step build) on the current
  stream.  Uniform draws come from a device Philox stream keyed by (seed, call counter) so the
  whole thing is CUDA-graph replayable; `uniforms=` lets tests inject the draws.
  """

  def __init__(self, table: Table, batch_size: int, seed: int = 0, stratified: bool = True,
               sequence_length=None, time_major: bool = False):
    import torch
    self.table, self.B, self.seed, self.stratified = table, int(batch_size), int(seed), bool(stratified)
    dev = torch.device('cuda', table.device)
    table._ensure()
    B = self.B
    self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
    self.u = torch.empty(B, dtype=torch.float32, device=dev)
    self.idx = torch.empty(B, dtype=torch.int64, device=dev)
    self.keys = torch.empty(B, dtype=torch.uint64, device=dev)
    self.prob = torch.empty(B, dtype=torch.float32, device=dev)
    # o_tm1 and o_t are the two halves of ONE [2B, obs_bytes] buffer: a learner can run its network over both batches
    # in a single pass (the online network sees o_tm1 and o_t, dqn/learning.py:123,125)
    self.sequence_length = int(sequence_length) if sequence_length else None
    self.time_major = bool(time_major)
    if table.is_sequence:
      # items are sequences (SURVEY §8f-3): [B][T] rows of whole steps ([T][B] with time_major, the layout
      # `tf2_utils.batch_to_sequence` produces for the recurrent learners, r2d2/learning.py:115)
      if not self.sequence_length:
        raise ValueError('a sequence table needs make_reverb_dataset(sequence_length=...)')
      T = self.sequence_length
      lead = (T, B) if self.time_major else (B, T)
      self.seq_obs = torch.empty(lead + (max(table.obs_packer.nbytes, 1),), dtype=torch.uint8, device=dev)
      self.seq_act = torch.empty(lead + (max(table.act_packer.nbytes, 1),), dtype=torch.uint8, device=dev)
      self.seq_rew = torch.empty(lead, dtype=torch.float32, device=dev)
      self.seq_disc = torch.empty(lead, dtype=torch.float32, device=dev)
      return
    self.o_both = torch.empty((2 * B, max(table.obs_packer.nbytes, 1)), dtype=torch.uint8, device=dev)
    self.o_tm1, self.o_t = self.o_both[:B], self.o_both[B:]
    self.a_tm1 = torch.empty((B, max(table.act_packer.nbytes, 1)), dtype=torch.uint8, device=dev)
    self.R = torch.empty(B, dtype=torch.float32, device=dev)
    self.D = torch.empty(B, dtype=torch.float32, device=dev)

  def sample_raw(self, uniforms=None):
    """Runs K1 + K3 into the dataset's static buffers (no host sync, graph-capturable)."""
    self.sample_only(uniforms)
    self.gather_only()

  def sample_only(self, uniforms=None, bump: bool = True):
    """K1: uniforms -> item indices, keys and probabilities (static buffers).  Without `uniforms` the draws are K1's own
    Philox stream keyed by (seed, call counter) -- the values `b200rl_uniform` would write, also stored in `self.u` -- and
    the counter advances afterwards (`bump=False`: the caller advances it, e.g. fused into the end of a learner step)."""
    stream = _capi.current_stream()
    if uniforms is None:
      _capi.call('b200rl_replay_sample_philox', self.table.handle, self.B, self.seed, _capi.ptr(self.counter),
                 int(self.stratified), _capi.ptr(self.u), _capi.ptr(self.idx), _capi.ptr(self.keys), _capi.ptr(self.prob), stream)
      if bump:
        _capi.call('b200rl_step_increment', _capi.ptr(self.counter), stream)
      return
    self.u.copy_(uniforms)
    self.table.sample_into(self.u, self.idx, self.keys, self.prob, self.stratified)

  def gather_only(self, rows=None):
    """K3: the sampled items' transitions (n-step return and discount built on the fly).  rows = (rows_tm1_ptr,
    rows_t_ptr, conv geometry): the frames are also written into the first conv layer's bf16 row images."""
    if self.table.is_sequence:
      _capi.call('b200rl_replay_gather_sequences', self.table.handle, self.B, _capi.ptr(self.idx), self.sequence_length,
                 int(self.time_major), _capi.ptr(self.seq_obs), _capi.ptr(self.seq_act), _capi.ptr(self.seq_rew),
                 _capi.ptr(self.seq_disc), _capi.current_stream())
      return
    if rows is not None:
      self.table.gather_rows_into(self.idx, self.o_tm1, self.a_tm1, self.R, self.D, self.o_t, *rows)
    else:
      self.table.gather_into(self.idx, self.o_tm1, self.a_tm1, self.R, self.D, self.o_t)

  def _sequence_sample(self, table_size: Optional[int] = None) -> ReplaySample:
    """data = the table's `Step` nest with leaves [B, T, ...] ([T, B, ...] when time_major); info fields are tiled over
    the time axis like `reverb.ReplayDataset(sequence_length=T)` does (r2d2/learning.py:172-173 reads `keys[:, 0]`)."""
    import torch
    t, T = self.table, self.sequence_length
    action, start, extras = t.act_packer.unpack_batch(self.seq_act)
    data = type(t.signature)(observation=t.obs_packer.unpack_batch(self.seq_obs), action=action, reward=self.seq_rew,
                             discount=self.seq_disc, start_of_episode=start, extras=extras)
    tile = (lambda x: x.unsqueeze(0).expand(T, -1)) if self.time_major else (lambda x: x.unsqueeze(1).expand(-1, T))
    prob64 = self.prob.to(torch.float64)
    if t.alpha > 0:
      mass = torch.as_tensor(_MassView(t.mass_ptr()), device=self.prob.device).to(torch.float64)
      priority = (prob64 * (t.shard_count * mass)).pow(1.0 / t.alpha)
    else:
      priority = torch.ones_like(prob64)
    size = t.size if table_size is None else table_size
    info = SampleInfo(key=tile(self.keys), probability=tile(prob64),
                      table_size=tile(torch.full((self.B,), size, dtype=torch.int64, device=self.prob.device)),
                      priority=tile(priority))
    return ReplaySample(info=info, data=data)

  def as_sample(self, table_size: Optional[int] = None) -> ReplaySample:
    import torch
    t = self.table
    if t.is_sequence:
      return self._sequence_sample(table_size)
    act = t.act_packer.unpack_batch(self.a_tm1)
    extras = None
    if t.has_extras:
      act, extras = act
    data = (t.obs_packer.unpack_batch(self.o_tm1), act, self.R, self.D, t.obs_packer.unpack_batch(self.o_t))
    if extras is not None:
      data = data + (extras,)
    size = t.size if table_size is None else table_size
    # SampleInfo dtypes as in `acme/testing/fakes.py:251-259` (u64 key, f64 probability, i64 table_size, f64 priority).
    # The tree stores priority^alpha in fp32 (that is what K1 reads): the reported probability is that fp32 quotient
    # widened, and the priority is recovered from it (leaf = probability * shards * shard mass; priority =
    # leaf^(1/alpha)).  With alpha = 0 (Uniform) every stored weight is 1 and the raw priority is not retained: 1.0.
    prob64 = self.prob.to(torch.float64)
    if t.alpha > 0:
      mass = torch.as_tensor(_MassView(t.mass_ptr()), device=self.prob.device).to(torch.float64)
      priority = (prob64 * (t.shard_count * mass)).pow(1.0 / t.alpha)
    else:
      priority = torch.ones_like(prob64)
    info = SampleInfo(key=self.keys, probability=prob64,
                      table_size=torch.full((self.B,), size, dtype=torch.int64, device=self.prob.device),
                      priority=priority)
    return ReplaySample(info=info, data=data)

  def __iter__(self):
    return self

  def __next__(self) -> ReplaySample:
    t = self.table
    t.flush()
    if not t.can_sample(self.B):
      raise RuntimeError('replay table has fewer items than its MinSize limiter requires')
    self.sample_raw()
    return self.as_sample()


def make_reverb_dataset(server_address=None, client: Optional[Client] = None, batch_size: int = 256,
                        prefetch_size: Optional[int] = None, sequence_length: Optional[int] = None,
                        extra_spec=None, environment_spec=None, table: str = DEFAULT_PRIORITY_TABLE,
                        seed: int = 0, stratified: bool = True, time_major: bool = False, **unused) -> ReplayDataset:
  """acme/datasets/reverb.py:36-139.  `prefetch_size` is accepted and ignored: batches are built
  synchronously in HBM, so samples are never stale with respect to priorities."""
  if client is None:
    if server_address is None:
      raise ValueError('either client or server_address must be given')
    client = Client(server_address)
  return ReplayDataset(client.table(table), batch_size, seed=seed, stratified=stratified,
                       sequence_length=sequence_length, time_major=time_major)
