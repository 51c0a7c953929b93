"""Multi-GPU sharding: one process per GPU, envs partitioned by index.

Environments never interact (one `Engine`/`Plot` per env upstream,
engine.py:216), so the step path shards with NO data-path collective: rank r
owns the contiguous block of env indices `shard_range(global_batch, r, world)`
together with their action stream and RNG states (seeded by GLOBAL env index,
so a sharded run reproduces the single-GPU run env for env).  The only
exchange is the optional hand-off of the per-step outputs to every rank:
`Handoff` packs each env's observation view + reward + discount + done into one
record on the device (`pcl_pack_handoff`) and moves everything with ONE NCCL
all-gather per step over NVLink/NVSwitch; `allgather_outputs` is the plain
one-collective-per-tensor form.
"""

import numpy as np


def shard_range(global_batch, rank, world):
  """Contiguous block partition: (first global env index, count) of `rank`."""
  if not 0 <= rank < world:
    raise ValueError('rank %d outside world of %d' % (rank, world))
  base, extra = divmod(global_batch, world)
  count = base + (1 if rank < extra else 0)
  first = rank * base + min(rank, extra)
  return first, count


def make_shard_engine(games, global_batch, rank, world, device, **kwargs):
  """`BatchedEngine` for this rank's block of a `global_batch`-env job.

  games[i] is the level of GLOBAL env i (mod len(games)): the local list is
  rotated so that local env e maps to global env first + e.  With
  cycle_levels=True every shard keeps the whole pool and steps through it by the
  GLOBAL batch, so the shards together walk it as one engine would."""
  from pycolab_b200 import batched
  first, count = shard_range(global_batch, rank, world)
  n = len(games)
  if kwargs.get('cycle_levels'):
    kwargs.setdefault('level_stride', global_batch)
    return batched.BatchedEngine(list(games), batch=count, device=device, env_offset=first,
                                 **kwargs)
  local = [games[(first + i) % n] for i in range(min(n, count))] if n > 1 else games
  return batched.BatchedEngine(local, batch=count, device=device, env_offset=first,
                               **kwargs)


def allgather_outputs(tensors, global_batch, group=None):
  """All-gather per-env output tensors (dim 0 = local envs) to [global_batch, ...].

  Shards may differ by one env when world does not divide global_batch; every
  rank pads to the largest shard, gathers, then drops the padding."""
  import torch
  import torch.distributed as dist
  world = dist.get_world_size(group)
  counts = [shard_range(global_batch, r, world)[1] for r in range(world)]
  biggest = max(counts)
  out = []
  for t in tensors:
    pad = t
    if t.shape[0] < biggest:
      pad = torch.cat([t, t.new_zeros((biggest - t.shape[0],) + tuple(t.shape[1:]))])
    pad = pad.contiguous()
    gathered = pad.new_empty((world * biggest,) + tuple(t.shape[1:]))
    dist.all_gather_into_tensor(gathered, pad, group=group)
    if all(c == biggest for c in counts):
      out.append(gathered)
    else:
      pieces = [gathered[r * biggest: r * biggest + counts[r]] for r in range(world)]
      out.append(torch.cat(pieces))
  return out


def handoff_record_bytes(view_bytes):
  """include/pcl.h: PCL_HANDOFF_RECORD_BYTES."""
  return ((view_bytes + 3) & ~3) + 12


def unpack_handoff(records, view_shape):
  """Views into packed hand-off records u8 [N, record_bytes] (no copies):
  (view u8 [N, *view_shape], reward i32 [N], discount f32 [N], done u8 [N],
  has_reward u8 [N]).  record_bytes may exceed PCL_HANDOFF_RECORD_BYTES (the fused
  path pads records to a multiple of 16)."""
  import torch
  view_bytes = 1
  for d in view_shape:
    view_bytes *= int(d)
  word = ((view_bytes + 3) & ~3) // 4
  n = records.shape[0]
  assert records.dtype == torch.uint8 and records.shape[1] >= handoff_record_bytes(view_bytes)
  assert records.shape[1] % 4 == 0
  view = records[:, :view_bytes].reshape((n,) + tuple(view_shape))
  return (view, records.view(torch.int32)[:, word], records.view(torch.float32)[:, word + 1],
          records[:, 4 * word + 8], records[:, 4 * word + 9])


class Handoff(object):
  """The per-step hand-off of one rank's shard to every rank (SURVEY.md 8e) with a
  single collective: pack on the device, one `all_gather_into_tensor`, unpack as
  views.  Buffers are allocated once."""

  def __init__(self, engine, view_shape, global_batch, group=None):
    import torch
    import torch.distributed as dist
    self.engine, self.group = engine, group
    self.view_shape = tuple(int(d) for d in view_shape)
    self.view_bytes = int(np.prod(self.view_shape))
    world = dist.get_world_size(group)
    self.counts = [shard_range(global_batch, r, world)[1] for r in range(world)]
    assert self.counts[dist.get_rank(group)] == engine.batch
    self.biggest = max(self.counts)
    rec = handoff_record_bytes(self.view_bytes)
    self.packed = torch.zeros((self.biggest, rec), dtype=torch.uint8, device=engine.device)
    self.gathered = torch.empty((world * self.biggest, rec), dtype=torch.uint8,
                                device=engine.device)

  def gather(self, view):
    """`view`: u8 [local envs, *view_shape] (contiguous), e.g. `engine.crop(spec)`."""
    self.engine.pack_handoff(view, self.packed)
    return self.exchange()

  def exchange(self):
    import torch
    import torch.distributed as dist
    dist.all_gather_into_tensor(self.gathered, self.packed, group=self.group)
    records = self.gathered
    if any(c != self.biggest for c in self.counts):       # drop the padding of short shards
      records = torch.cat([records[r * self.biggest: r * self.biggest + c]
                           for r, c in enumerate(self.counts)])
    return unpack_handoff(records, self.view_shape)


class PeerHandoff(object):
  """`Handoff` without a collective call: the gather buffers live in symmetric
  memory (every rank maps every peer's buffer), the pack kernel stores each record
  into ALL of them over NVLink (`pcl_pack_handoff_peers`), and one device-side
  barrier per step tells the consumers that every rank's records have landed.
  Two buffers alternate, so a step may overwrite only what was consumed (in
  stream order) before the previous step's barrier."""

  def __init__(self, engine, view_shape, global_batch, group=None):
    import torch
    import torch.distributed as dist
    import torch.distributed._symmetric_memory as symm_mem
    group = group if group is not None else dist.group.WORLD
    self.engine = engine
    self.view_shape = tuple(int(d) for d in view_shape)
    self.view_bytes = int(np.prod(self.view_shape))
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    self.counts = [shard_range(global_batch, r, world)[1] for r in range(world)]
    assert self.counts[rank] == engine.batch
    self.biggest = max(self.counts)
    self.rows, self.rec = world * self.biggest, handoff_record_bytes(self.view_bytes)
    self.first_row = rank * self.biggest
    half = self.rows * self.rec
    self.buffer = symm_mem.empty(2 * half, dtype=torch.uint8, device=engine.device)
    self.buffer.zero_()
    self.handle = symm_mem.rendezvous(self.buffer, group)
    self.peer_ptrs = [[int(p) + k * half for p in self.handle.buffer_ptrs] for k in (0, 1)]
    self.halves = [self.buffer[k * half:(k + 1) * half].view(self.rows, self.rec)
                   for k in (0, 1)]
    self.step = 0
    self.handle.barrier(channel=0)            # everyone's buffers exist and are zeroed

  def gather(self, view):
    k = self.step & 1
    self.step += 1
    self.engine.pack_handoff_peers(view, self.peer_ptrs[k], self.first_row)
    self.handle.barrier(channel=0)            # all ranks' stores have been issued and finished
    records = self.halves[k]
    if any(c != self.biggest for c in self.counts):
      import torch
      records = torch.cat([records[r * self.biggest: r * self.biggest + c]
                           for r, c in enumerate(self.counts)])
    return unpack_handoff(records, self.view_shape)


class FusedHandoff(object):
  """The per-step hand-off as ONE kernel per rank (`pcl_crop_handoff`): the cropper,
  the record packing, the stores into every rank's gather buffer over NVLink (or one
  NVLS multicast store) and the cross-GPU flag barrier.  Gather buffers and flag
  arrays live in symmetric memory; nothing from a collective library runs per step
  and the launch can be captured in a CUDA graph (the step counter is on the
  device).  With a single rank it degenerates to crop + pack into a local buffer.

  lag=1 is the split-phase form: the kernel of step s signals s but waits only for
  step s - 1 of the peers, so the cross-GPU wait is off the critical path; `gather()`
  then returns the records of the PREVIOUS step (None on the first call) and `flush()`
  — a host-level barrier — completes the last one.  Three buffer parts alternate.

  signal_kernel=True (default) publishes and waits in a second one-warp kernel behind
  the records kernel instead of fencing in each of its thread blocks (measured faster)."""

  def __init__(self, engine, crop_spec, global_batch, group=None, multicast=True, lag=0,
               signal_kernel=True):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from pycolab_b200 import _lib
    self.engine, self.crop_spec = engine, crop_spec
    self.view_shape = (int(crop_spec.rows), int(crop_spec.cols))
    self.view_bytes = self.view_shape[0] * self.view_shape[1]
    if dist.is_available() and dist.is_initialized():
      group = group if group is not None else dist.group.WORLD
      world, rank = dist.get_world_size(group), dist.get_rank(group)
    else:
      world, rank = 1, 0
    self.counts = [shard_range(global_batch, r, world)[1] for r in range(world)]
    assert self.counts[rank] == engine.batch
    self.biggest = max(self.counts)
    self.rows = world * self.biggest
    self.rec = (handoff_record_bytes(self.view_bytes) + 15) & ~15
    self.first_row = rank * self.biggest
    self.lag = int(lag)
    self.n_bufs = 3 if self.lag else 2
    half = self.rows * self.rec
    flag_bytes = 256
    total = self.n_bufs * half + flag_bytes
    self.handle = None
    mc_ptr = 0
    if world > 1:
      import torch.distributed._symmetric_memory as symm_mem
      self.buffer = symm_mem.empty(total, dtype=torch.uint8, device=engine.device)
      self.buffer.zero_()
      self.handle = symm_mem.rendezvous(self.buffer, group)
      bases = [int(p) for p in self.handle.buffer_ptrs]
      if multicast:
        try:
          mc_ptr = int(getattr(self.handle, 'multicast_ptr', 0) or 0)
        except Exception:           # noqa: BLE001 - no NVLS on this box: unicast stores
          mc_ptr = 0
    else:
      self.buffer = torch.zeros(total, dtype=torch.uint8, device=engine.device)
      bases = [self.buffer.data_ptr()]
    self.transport = 'NVLS multicast stores' if mc_ptr else (
        'peer-to-peer stores' if world > 1 else 'local stores (single rank)')
    self.local = torch.zeros(2, dtype=torch.int32, device=engine.device)
    st = _lib.HandoffState()
    st.n_peers, st.rank, st.record_bytes = world, rank, self.rec
    st.rows, st.first_row = self.rows, self.first_row
    for i, b in enumerate(bases):
      st.d_peer_base[i] = b
      st.d_peer_flags[i] = b + self.n_bufs * half
    st.d_multicast = mc_ptr or None
    st.d_local = self.local.data_ptr()
    st.n_bufs = self.n_bufs
    st.mode = ((_lib.HANDOFF_LAG if self.lag else 0) |
               (_lib.HANDOFF_SIGNAL_KERNEL if signal_kernel else 0))
    self.signal_kernel = bool(signal_kernel)
    self._state = st
    self.halves = [self.buffer[k * half:(k + 1) * half].view(self.rows, self.rec)
                   for k in range(self.n_bufs)]
    self.crop_state = engine.new_crop_state()
    self.step = 0
    torch.cuda.synchronize(engine.device)
    if self.handle is not None:
      self.handle.barrier(channel=0)          # everyone's buffers exist and are zeroed

  def gather(self):
    """Crop the engine's last boards and exchange: (view u8 [N, rows, cols], reward,
    discount, done, has_reward) of ALL ranks' envs, views into this rank's buffer.
    With lag=1: of the PREVIOUS step (None on the first call)."""
    k = self.step % self.n_bufs
    self.step += 1
    self.engine.crop_handoff(self.crop_spec, self.crop_state, self._state)
    if self.lag:
      if self.step == 1:
        return None
      k = (self.step - 2) % self.n_bufs
    return self._unpack(k)

  def _unpack(self, k):
    records = self.halves[k]
    if any(c != self.biggest for c in self.counts):
      import torch
      records = torch.cat([records[r * self.biggest: r * self.biggest + c]
                           for r, c in enumerate(self.counts)])
    return unpack_handoff(records, self.view_shape)

  def flush(self):
    """lag=1: make the LAST step's records complete everywhere (stream drained + a
    host-level barrier: every rank's kernel has retired, and a retired kernel's peer
    stores are visible) and return them."""
    import torch
    torch.cuda.synchronize(self.engine.device)
    if self.handle is not None:
      self.handle.barrier(channel=0)
    # the DEVICE's step count names the part (CUDA-graph replays advance it without
    # passing through gather())
    done = int(self.local[0].item())
    self.step = done
    return self._unpack((done - 1) % self.n_bufs)
