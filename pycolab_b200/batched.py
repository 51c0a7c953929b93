"""`BatchedEngine`: B independent pycolab environments stepped in lockstep on one GPU.

The batched counterpart of the reference's one-`Engine`-per-env loop
(engine.py:520-639): `its_showtime()` / `play(actions)` keep their meaning,
vectorised over the env axis.  State lives in HBM as a struct-of-arrays
(include/pcl.h `pcl_state`); PyTorch is used only to own the device buffers
and the stream.  Every step is ONE fused CUDA kernel launched through the
C ABI (`pcl_step`); there is no CPU path.
"""

import ctypes as C

import numpy as np

from pycolab_b200 import _lib
from pycolab_b200 import lowering


def _torch():
  import torch
  return torch


class StepResult(object):
  """(board, reward, has_reward, discount, done) of one batched step.

  board: u8 [B, rows, cols] view into the engine-owned output buffer (valid
  until the next step — copy to keep, as upstream rendering.py:55-63).
  reward: i32 [B] with has_reward u8 [B] == 0 where the reference returns None.
  discount: f32 [B].  done: u8 [B] (Engine.game_over).
  """
  __slots__ = ('board', 'reward', 'has_reward', 'discount', 'done')

  def __init__(self, board, reward, has_reward, discount, done):
    self.board, self.reward, self.has_reward = board, reward, has_reward
    self.discount, self.done = discount, done

  def __iter__(self):            # (observation, reward, discount) like Engine.play
    return iter((self.board, self.reward, self.discount))


class BatchedEngine(object):

  def __init__(self, games, batch=None, device=0, auto_reset=True, rng_seed=0,
               env_offset=0, rng_states=None, share_levels=True, cycle_levels=False,
               level_stride=None):
    """games: list of lowered games (`lowering.LoweredGame`) or set-up `Engine`s.
    Env e uses games[e % len(games)]; with a single game the static level data
    (backdrop, immutable patterns, reset templates) is shared by all envs.
    env_offset: global index of this shard's env 0 (per-env RNG streams are
    seeded rng_seed + global env index — NumPy RandomState(seed) or, for games that
    draw from Python's `random`, random.Random(seed)); rng_states: explicit u32 [B, 625]
    (False: bind no RNG, for programs that can take their draws from the templates)
    MT19937 states (624 key words + position) instead of seeds.
    share_levels=False stores the static level data once PER ENV instead of once
    per level (the reference's layout: every Engine owns its backdrop).
    cycle_levels=True (Box-World only, more than one level, shared levels): the pool
    is walked instead of pinned: env e starts on level (env_offset + e) % n and every
    auto-reset moves it on by `level_stride` levels (default: the batch), so envs
    e, e + B, e + 2B, ... cover the whole pool.  A masked reset() restarts the same
    level."""
    torch = _torch()
    self._lib = _lib.load()
    games = [g if isinstance(g, lowering.LoweredGame) else lowering.lower(g)
             for g in (games if isinstance(games, (list, tuple)) else [games])]
    sig = games[0].signature()
    for g in games[1:]:
      if g.signature() != sig:
        raise ValueError('all games of one BatchedEngine must share one structure')
    self.game = g0 = games[0]
    self.batch = B = int(batch if batch is not None else len(games))
    if cycle_levels:
      if g0.program != _lib.PROG_BOX_WORLD:
        raise ValueError('cycle_levels is supported for the box_world program only')
      if len(games) < 2:
        raise ValueError('cycle_levels needs more than one level')
      if not share_levels:
        raise ValueError('cycle_levels needs share_levels=True (envs change level)')
      level_stride = B if level_stride is None else int(level_stride)
      if level_stride < 1:
        raise ValueError('level_stride must be positive')
    elif level_stride is not None:
      raise ValueError('level_stride is meaningful with cycle_levels only')
    self.cycle_levels = bool(cycle_levels)
    if not torch.cuda.is_available():
      raise _lib.PclLibraryError('CUDA device required: pycolab_b200 has no CPU path')
    self.device = torch.device('cuda', device)
    self.auto_reset = bool(auto_reset)
    self.rows, self.cols, self.pitch = g0.rows, g0.cols, g0.pitch
    self.sprite_chars, self.drape_chars = g0.sprite_chars, g0.drape_chars
    self.chars = ''.join(sorted(set(g0.sprite_chars + g0.drape_chars + g0.backdrop_chars)))
    n = len(games)
    shared = (n == 1)
    dev = self.device

    def tiled(arrays, dtype):
      """Static data: ONE copy per level ([n_levels, ...]); envs find theirs
      through the level index (pcl_state.d_level), or share the single copy."""
      stacked = np.stack([np.ascontiguousarray(a).astype(dtype) for a in arrays])
      return torch.from_numpy(stacked).to(dev)

    def per_env(arrays, dtype):
      stacked = np.stack([np.ascontiguousarray(a).astype(dtype) for a in arrays])
      t = torch.from_numpy(stacked).to(dev)
      reps = (B + n - 1) // n
      return t.repeat((reps,) + (1,) * (t.dim() - 1))[:B].contiguous()

    def bstride(t):
      return 0 if t.shape[0] == 1 else t[0].numel()

    if not share_levels:
      tiled, shared = per_env, True     # every array env-indexed, no level table

    self._keep = []             # every tensor the handle points at
    st = _lib.State()
    self.level = None           # i32 [B]: which level each env plays
    if not shared:
      first = env_offset if cycle_levels else 0
      self.level = ((torch.arange(B, dtype=torch.int64, device=dev) + first) % n).to(
          torch.int32).contiguous()
      st.d_level = self.level.data_ptr()
    self.backdrop = tiled([g.backdrop for g in games], np.uint8)
    st.d_backdrop, st.backdrop_bstride = self.backdrop.data_ptr(), bstride(self.backdrop)
    self.patterns, self.bits = {}, {}
    self._keep_bits_init = {}
    for d in sorted(g0.patterns):
      arrays = [g.patterns[d].view(np.int32) for g in games]
      if g0.pattern_mutable[d]:
        init = tiled(arrays, np.int32)
        live = per_env(arrays, np.int32)
        st.d_pattern_init[d], st.pattern_init_bstride[d] = init.data_ptr(), bstride(init)
        self._keep.append(init)
      else:
        live = tiled(arrays, np.int32)
      self.patterns[d] = live
      st.d_pattern[d] = live.data_ptr()
      st.pattern_bstride[d] = bstride(live) if not g0.pattern_mutable[d] else live[0].numel()
    for d in sorted(g0.bits):
      arrays = [g.bits[d].view(np.int32) for g in games]
      init = tiled(arrays, np.int32)
      live = per_env(arrays, np.int32)
      self.bits[d] = live
      self._keep.append(init)
      self._keep_bits_init[d] = init
      st.d_bits[d], st.bits_bstride[d] = live.data_ptr(), live[0].numel()
      st.d_bits_init[d], st.bits_init_bstride[d] = init.data_ptr(), bstride(init)
    self.sprites = per_env([g.sprites for g in games], np.int32)
    self.drapes = per_env([g.drapes for g in games], np.int32)
    self.plot = per_env([g.plot for g in games], np.int32)
    # Live records start "game over" so the first pcl_reset builds every env.
    self._sprites_init = tiled([g.sprites for g in games], np.int32)
    self._drapes_init = tiled([g.drapes for g in games], np.int32)
    self._plot_init = tiled([g.plot for g in games], np.int32)
    st.d_sprites, st.d_sprites_init = self.sprites.data_ptr(), self._sprites_init.data_ptr()
    st.sprites_init_bstride = bstride(self._sprites_init)
    st.d_drapes, st.d_drapes_init = self.drapes.data_ptr(), self._drapes_init.data_ptr()
    st.drapes_init_bstride = bstride(self._drapes_init)
    st.d_plot, st.d_plot_init = self.plot.data_ptr(), self._plot_init.data_ptr()
    st.plot_init_bstride = bstride(self._plot_init)
    self.z_order = None
    if g0.dynamic_z:
      zs = [np.frombuffer(g.z_order.encode('ascii'), dtype=np.uint8) for g in games]
      self.z_order = per_env(zs, np.uint8)
      self._z_init = tiled(zs, np.uint8)
      st.d_z_order, st.d_z_order_init = self.z_order.data_ptr(), self._z_init.data_ptr()
      st.z_order_init_bstride = bstride(self._z_init)
    self.groups = None          # scrolling groups >= 1 (group 0 is in the plot record)
    if len(g0.scroll_groups) > 1:
      self.groups = per_env([g.group_records for g in games], np.int32)
      self._groups_init = tiled([g.group_records for g in games], np.int32)
      st.d_groups, st.d_groups_init = self.groups.data_ptr(), self._groups_init.data_ptr()
      st.groups_init_bstride = bstride(self._groups_init)
    self.actions_per_env = (len(g0.sprite_chars) + len(g0.drape_chars) +
                            2 * _lib.FIXTURE_DIRECTIVES
                            if g0.program == _lib.PROG_FIXTURE else 1)
    self.rng = None
    if g0.needs_rng and rng_states is not False:
      if rng_states is not None:
        states = np.ascontiguousarray(rng_states, dtype=np.uint32).reshape(B, _lib.MT_WORDS)
      elif getattr(g0, 'rng_kind', 'numpy') == 'python':
        # Python's `random` (apprehend.py:103): the 625 words of Random(seed).getstate()
        import random as _random
        states = np.empty((B, _lib.MT_WORDS), dtype=np.uint32)
        for e in range(B):
          states[e] = _random.Random(rng_seed + env_offset + e).getstate()[1]
      else:
        states = np.empty((B, _lib.MT_WORDS), dtype=np.uint32)
        for e in range(B):
          _, key, pos, _, _ = np.random.RandomState(rng_seed + env_offset + e).get_state()
          states[e, :624] = key
          states[e, 624] = pos
      self.rng = torch.from_numpy(states.view(np.int32)).to(dev)
      st.d_rng = self.rng.data_ptr()
    self._state = st

    # Outputs.
    self._board = torch.zeros((B, self.rows, self.pitch), dtype=torch.uint8, device=dev)
    self.reward = torch.zeros((B,), dtype=torch.int32, device=dev)
    self.has_reward = torch.zeros((B,), dtype=torch.uint8, device=dev)
    self.discount = torch.ones((B,), dtype=torch.float32, device=dev)
    self.done = torch.zeros((B,), dtype=torch.uint8, device=dev)
    self._out = _lib.Outputs(self._board.data_ptr(), self.reward.data_ptr(),
                             self.has_reward.data_ptr(), self.discount.data_ptr(),
                             self.done.data_ptr())
    self._actions = torch.zeros((B * self.actions_per_env,), dtype=torch.int32, device=dev)
    self._host = None           # pinned staging for play_host() / play_host_async(), per slot
    self._slot_shape = {}
    self._crop_dev = None
    self._crop_out = None
    self._attached = None       # attach_cropper: (spec, state, out, runs inside the step kernel)

    self._spec = g0.make_spec(self.auto_reset)
    if cycle_levels:
      self._spec.program_arg[1], self._spec.program_arg[2] = level_stride, n
    handle = C.c_void_p()
    _lib.check(self._lib.pcl_create(C.byref(self._spec), B, self.device.index,
                                    C.byref(handle)), 'pcl_create')
    self._h = handle
    _lib.check(self._lib.pcl_bind_state(self._h, C.byref(self._state)), 'pcl_bind_state')
    self._showtime = False

  # ---------------------------------------------------------------- running
  def _stream(self):
    return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

  @property
  def board(self):
    """u8 [B, rows, cols] view of the last rendered boards."""
    return self._board[:, :, :self.cols]

  def _result(self):
    return StepResult(self.board, self.reward, self.has_reward, self.discount, self.done)

  def its_showtime(self):
    """Engine.its_showtime() for every env (engine.py:520-581)."""
    if self._showtime:
      raise RuntimeError('its_showtime should not be called after its_showtime() has '
                         'been called')
    self._showtime = True
    _lib.check(self._lib.pcl_reset(self._h, None, C.byref(self._out), self._stream()),
               'pcl_reset', self._h)
    self._after_step()
    return self._result()

  def reset(self, env_mask=None):
    """Rebuild the selected envs (u8/bool [B] device tensor; None = all) and run
    their its_showtime() frame; other envs are untouched."""
    self._showtime = True
    mask = None
    if env_mask is not None:
      mask = env_mask.to(device=self.device, dtype=_torch().uint8).contiguous()
    _lib.check(self._lib.pcl_reset(self._h, None if mask is None else mask.data_ptr(),
                                   C.byref(self._out), self._stream()), 'pcl_reset', self._h)
    self._after_step()
    return self._result()

  def play(self, actions):
    """Engine.play(actions) for every env (engine.py:583-639).

    actions: int32 [B] device tensor (or anything torch.as_tensor accepts).
    With auto_reset, an env that was game-over is rebuilt instead and its
    action is ignored; without it such envs stay frozen (upstream raises)."""
    if not self._showtime:
      raise RuntimeError('play() cannot be called until the Engine is placed in "play '
                         'mode" via the its_showtime() method.')
    torch = _torch()
    if not (torch.is_tensor(actions) and actions.is_cuda and
            actions.dtype == torch.int32 and actions.is_contiguous()):
      actions = torch.as_tensor(actions, dtype=torch.int32).to(self.device).contiguous()
    if actions.numel() != self.batch * self.actions_per_env:
      raise ValueError('expected %d action words, got %d' % (
          self.batch * self.actions_per_env, actions.numel()))
    _lib.check(self._lib.pcl_step(self._h, actions.data_ptr(), C.byref(self._out),
                                  self._stream()), 'pcl_step', self._h)
    self._after_step()
    return self._result()

  def run(self, actions):
    """T back-to-back steps; actions int32 [T, B] on the device."""
    torch = _torch()
    assert actions.is_cuda and actions.dtype == torch.int32 and actions.is_contiguous()
    assert actions.dim() >= 2 and actions[0].numel() == self.batch * self.actions_per_env
    _lib.check(self._lib.pcl_run(self._h, actions.data_ptr(), int(actions.shape[0]),
                                 C.byref(self._out), self._stream()), 'pcl_run', self._h)
    return self._result()

  def _host_buffers(self, slot, view_shape):
    """Pinned staging of one pipeline slot (allocated on first use)."""
    torch = _torch()
    key = (slot, tuple(view_shape))
    if self._host is None:
      self._host = {}
    if key not in self._host:
      pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory()
      t = dict(actions=pin((self.batch * self.actions_per_env,), torch.int32),
               view=pin(tuple(view_shape), torch.uint8),
               reward=pin((self.batch,), torch.int32), has_reward=pin((self.batch,), torch.uint8),
               discount=pin((self.batch,), torch.float32), done=pin((self.batch,), torch.uint8))
      self._host[key] = (t, {k: v.numpy() for k, v in t.items()})
    return self._host[key]

  def play_host(self, actions, want_board=True):
    """Host-buffer step through `pcl_step_host`: int32 [B] numpy actions in,
    numpy (board [B, rows, pitch] padded, reward, has_reward, discount, done)
    views of pinned host buffers out; synchronises."""
    h, n = self._host_buffers(0, (self.batch, self.rows, self.pitch))
    n['actions'][:] = np.asarray(actions, dtype=np.int32).reshape(-1)
    _lib.check(self._lib.pcl_step_host(
        self._h, h['actions'].data_ptr(), self._actions.data_ptr(), C.byref(self._out),
        h['view'].data_ptr() if want_board else None, h['reward'].data_ptr(),
        h['has_reward'].data_ptr(), h['discount'].data_ptr(), h['done'].data_ptr(),
        self._stream()), 'pcl_step_host', self._h)
    return (n['view'][:, :, :self.cols], n['reward'], n['has_reward'], n['discount'],
            n['done'])

  def play_host_async(self, actions, slot=0, crop_spec=None, crop_state=None):
    """Pipelined host-buffer step (`pcl_step_host_async`): enqueue H2D(actions),
    the step (and, with `crop_spec`, the cropper) and the D2H of the outputs on
    the engine's copy stream, and return at once.  `host_wait(slot)` blocks until
    this call's results are valid and returns them.  With a crop spec only the
    cropped view u8 [B, rows, cols] crosses PCIe."""
    if not self._showtime:
      raise RuntimeError('play() cannot be called until its_showtime() has been called')
    if crop_spec is None:
      shape = (self.batch, self.rows, self.pitch)
    else:
      shape = (self.batch, crop_spec.rows, crop_spec.cols)
      att = getattr(self, '_attached', None)
      if (att is not None and att[3] and bytes(att[0]) == bytes(crop_spec) and
          (crop_state is None or crop_state.data_ptr() == att[1].data_ptr())):
        # this very cropper runs inside the step kernel: ship its view, launch nothing more
        self._crop_dev, crop_state = att[2], att[1]
      elif self._crop_dev is None or tuple(self._crop_dev.shape) != shape:
        self._crop_dev = _torch().empty(shape, dtype=_torch().uint8, device=self.device)
    h, n = self._host_buffers(slot, shape)
    n['actions'][:] = np.asarray(actions, dtype=np.int32).reshape(-1)
    _lib.check(self._lib.pcl_step_host_async(
        self._h, h['actions'].data_ptr(), self._actions.data_ptr(), C.byref(self._out),
        None if crop_spec is None else C.addressof(crop_spec),
        None if crop_spec is None else self._crop_dev.data_ptr(),
        None if crop_state is None else crop_state.data_ptr(),
        h['view'].data_ptr(), h['reward'].data_ptr(), h['has_reward'].data_ptr(),
        h['discount'].data_ptr(), h['done'].data_ptr(), int(slot), self._stream()),
        'pcl_step_host_async', self._h)
    self._slot_shape[slot] = shape

  def host_wait(self, slot=0):
    """Results of the `play_host_async` call that used `slot`: numpy views of its
    pinned buffers (view, reward, has_reward, discount, done)."""
    _lib.check(self._lib.pcl_host_wait(self._h, int(slot)), 'pcl_host_wait', self._h)
    _, n = self._host_buffers(slot, self._slot_shape[slot])
    view = n['view']
    if view.shape[1:] == (self.rows, self.pitch):
      view = view[:, :, :self.cols]
    return view, n['reward'], n['has_reward'], n['discount'], n['done']

  # ------------------------------------------------------------- accessors
  def curtain(self, char):
    """Drape.curtain of every env as bool [B, rows, cols] (things.py:213-217)."""
    if self.game.program == _lib.PROG_BOX_WORLD:
      # every key, lock and gem lives in the cell plane: byte = character | distractor bit
      return (self.plane()[:, :, :self.cols] & 0x7f) == ord(char)
    return self._curtain_bytes(self.drape_chars.index(char))[:, :, :self.cols].bool()

  def plane(self):
    """Box-World cell plane of every env, u8 [B, rows, pitch] (a view of the live
    state, see pcl.h PCL_PROG_BOX_WORLD)."""
    if self.game.program != _lib.PROG_BOX_WORLD:
      raise ValueError('only the box_world program keeps a cell plane')
    return self.bits[0].view(_torch().uint8)

  def _curtain_bytes(self, d):
    """Curtain of drape `d` as u8 [B, rows, pitch] (the pcl_export_curtain layout)."""
    torch = _torch()
    out = torch.empty((self.batch, self.rows, self.pitch), dtype=torch.uint8,
                      device=self.device)
    if self.game.program == _lib.PROG_WAREHOUSE:
      # JudgeDrape curtain = cells of boxes currently drawn as 'X'.
      out.zero_()
      nb = len(self.sprite_chars) - 1
      rec = self.sprites[:, :nb]
      on = rec[:, :, _lib.S_AUX0] != 0
      b, s = torch.nonzero(on, as_tuple=True)
      out[b, rec[b, s, _lib.S_ROW].long(), rec[b, s, _lib.S_COL].long()] = 1
    elif self.game.program == _lib.PROG_HELLO:
      # RollingDrape: the reset curtain shifted by the record's (AUX0, AUX1) counters.
      from pycolab_b200 import lowering
      if getattr(self, '_roll_base', None) is None:
        init = self._keep_bits_init[d].cpu().numpy().view(np.uint32)
        base = np.stack([lowering.unpack_rows(lvl, self.cols) for lvl in init])
        self._roll_base = torch.from_numpy(base.astype(np.uint8)).to(self.device)
      lvl = (self.level.long() if self.level is not None
             else torch.zeros(self.batch, dtype=torch.long, device=self.device))
      if self._roll_base.shape[0] == self.batch and self.level is None and self.batch > 1:
        lvl = torch.arange(self.batch, device=self.device)
      rr = (torch.arange(self.rows, device=self.device)[None, :] -
            self.drapes[:, d, _lib.D_AUX0].long()[:, None]) % self.rows
      cc = (torch.arange(self.cols, device=self.device)[None, :] -
            self.drapes[:, d, _lib.D_AUX1].long()[:, None]) % self.cols
      out.zero_()
      out[:, :, :self.cols] = self._roll_base[lvl[:, None, None], rr[:, :, None], cc[:, None, :]]
    elif self.game.program == _lib.PROG_APERTURE:
      # ApertureDrape curtain = the (at most two) cells of its `_apertures` list.
      out.zero_()
      for word in (_lib.D_AUX0, _lib.D_AUX1):
        cell = self.drapes[:, d, word]
        b = torch.nonzero(cell >= 0, as_tuple=True)[0]
        out[b, (cell[b] >> 16).long(), (cell[b] & 0xffff).long()] = 1
    else:
      _lib.check(self._lib.pcl_export_curtain(self._h, d, out.data_ptr(), self._stream()),
                 'pcl_export_curtain', self._h)
    return out

  def unoccluded_layers(self, chars=None):
    """Layers of `BaseUnoccludedObservationRenderer` (rendering.py:187-301) for
    every env: bool [B, len(chars), rows, cols], plane k = everywhere the owner of
    chars[k] places it, occluded or not.  Default chars: every character of the
    game, sorted (`self.chars`).  One kernel over the packed device state."""
    torch = _torch()
    chars = self.chars if chars is None else ''.join(chars)
    out = torch.empty((self.batch, len(chars), self.rows, self.pitch), dtype=torch.uint8,
                      device=self.device)
    _lib.check(self._lib.pcl_layers(self._h, chars.encode('ascii'), len(chars), out.data_ptr(),
                                    self._stream()), 'pcl_layers', self._h)
    return out[:, :, :, :self.cols].bool()

  def error_codes(self):
    torch = _torch()
    out = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
    _lib.check(self._lib.pcl_error_codes(self._h, out.data_ptr(), self._stream()),
               'pcl_error_codes', self._h)
    return out

  def launch_count(self):
    n = C.c_int64()
    _lib.check(self._lib.pcl_launch_count(self._h, C.byref(n)), 'pcl_launch_count')
    return n.value

  def new_crop_state(self):
    """Corner state of one cropper object: i32 [B, 4] (row, col, initialised,
    episode), zero = not yet initialised.  One per ScrollingCropper."""
    return _torch().zeros((self.batch, 4), dtype=_torch().int32, device=self.device)

  def attach_cropper(self, crop_spec, state=None, out=None):
    """Make every later its_showtime() / play() / run() also produce this cropper's view
    of the new boards — from inside the step kernel where the game program supports it
    (`pcl_attach_cropper`: no second launch), else by a crop launch after each step.
    Returns the u8 [B, rows, cols] tensor that always holds the latest views.
    `crop_spec=None` detaches."""
    torch = _torch()
    if crop_spec is None:
      _lib.check(self._lib.pcl_attach_cropper(self._h, None, None, None), 'pcl_attach_cropper')
      self._attached = None
      return None
    if out is None:
      out = torch.zeros((self.batch, crop_spec.rows, crop_spec.cols), dtype=torch.uint8,
                        device=self.device)
    if state is None:
      state = self.new_crop_state()
    status = self._lib.pcl_attach_cropper(self._h, C.byref(crop_spec), out.data_ptr(),
                                          state.data_ptr())
    if status == _lib.ERR_UNSUPPORTED:          # no epilogue in this program: crop after the step
      self._attached = (crop_spec, state, out, False)
    else:
      _lib.check(status, 'pcl_attach_cropper', self._h)
      self._attached = (crop_spec, state, out, True)
    return out

  def _after_step(self):
    att = getattr(self, '_attached', None)
    if att is not None and not att[3]:
      self.crop(att[0], state=att[1], out=att[2])

  def crop(self, crop_spec, state=None, out=None):
    """ScrollingCropper / FixedCropper .crop over the last boards: u8 [B, rows,
    cols].  `state` (from new_crop_state) keeps this cropper's window corners;
    None uses the single built-in slot in the plot record.  Without `out` the
    result lives in an engine-owned buffer of THIS cropper (one per `state`), valid
    until its next crop — copy to keep, as upstream (cropping.py:148-149)."""
    torch = _torch()
    shape = (self.batch, crop_spec.rows, crop_spec.cols)
    if out is None:
      # one engine-owned buffer per cropper (keyed by its corner state): two croppers
      # with the same window shape must not overwrite each other's view
      key = (shape, None if state is None else state.data_ptr())
      if self._crop_out is None:
        self._crop_out = {}
      if key not in self._crop_out:
        self._crop_out[key] = torch.empty(shape, dtype=torch.uint8, device=self.device)
      out = self._crop_out[key]
    state_ptr = None if state is None else state.data_ptr()
    if any(code < 0 for code in crop_spec.track):
      # A tracked drape's position is the median of its curtain cells: hand the
      # kernel the byte curtains (cropping.py:583-596).
      curtains, ptrs = [], (C.c_void_p * _lib.MAX_TRACK)()
      for i, code in enumerate(crop_spec.track):
        if code < 0:
          curtains.append(self._curtain_bytes(-code - 1))
          ptrs[i] = curtains[-1].data_ptr()
      _lib.check(self._lib.pcl_crop_tracking(self._h, C.byref(crop_spec),
                                             self._board.data_ptr(), out.data_ptr(), state_ptr,
                                             ptrs, self._stream()), 'pcl_crop_tracking', self._h)
    else:
      _lib.check(self._lib.pcl_crop(self._h, C.byref(crop_spec), self._board.data_ptr(),
                                    out.data_ptr(), state_ptr, self._stream()), 'pcl_crop', self._h)
    return out

  def pack_handoff(self, view, packed):
    """Pack `view` (u8 [B, ...], contiguous) with this step's reward / discount /
    done into `packed` u8 [>= B, PCL_HANDOFF_RECORD_BYTES] (dist.Handoff)."""
    torch = _torch()
    view_bytes = int(view[0].numel())
    assert view.dtype == torch.uint8 and view.is_contiguous() and view.shape[0] == self.batch
    assert packed.is_contiguous() and packed.shape[0] >= self.batch
    assert packed.shape[1] == ((view_bytes + 3) & ~3) + 12
    _lib.check(self._lib.pcl_pack_handoff(self._h, view.data_ptr(), view_bytes,
                                          C.byref(self._out), packed.data_ptr(),
                                          self._stream()), 'pcl_pack_handoff', self._h)
    return packed

  def pack_handoff_peers(self, view, peer_ptrs, first_row):
    """`pack_handoff` with the all-gather fused in: records go straight into row
    `first_row + env` of every rank's gather buffer (`peer_ptrs`: peer-mapped
    device pointers) over NVLink (dist.PeerHandoff)."""
    torch = _torch()
    assert view.dtype == torch.uint8 and view.is_contiguous() and view.shape[0] == self.batch
    ptrs = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
    _lib.check(self._lib.pcl_pack_handoff_peers(
        self._h, view.data_ptr(), int(view[0].numel()), C.byref(self._out), ptrs,
        len(peer_ptrs), int(first_row), self._stream()), 'pcl_pack_handoff_peers', self._h)

  def crop_handoff(self, crop_spec, crop_state, handoff_state):
    """ScrollingCropper.crop + record packing + the all-gather to every rank + the
    cross-GPU barrier as ONE kernel (`pcl_crop_handoff`, dist.FusedHandoff)."""
    _lib.check(self._lib.pcl_crop_handoff(
        self._h, C.byref(crop_spec), self._board.data_ptr(),
        None if crop_state is None else crop_state.data_ptr(), C.byref(self._out),
        C.byref(handoff_state), self._stream()), 'pcl_crop_handoff', self._h)

  # --- observation post-processors (rendering.py:304-661) over the whole batch
  def to_feature_array(self, layers, permute=None):
    """ObservationToFeatureArray: float32 one-hot planes, [B, C, rows, cols] (or
    the last three axes permuted)."""
    from pycolab_b200 import observers
    permute = observers.check_permute(permute, True, 'ObservationToFeatureArray')
    return observers.observe(self._lib, self._h, self._board, self.rows, self.cols,
                             observers.feature_table(layers), None, True, permute,
                             self._stream())

  def to_array(self, value_mapping, dtype=None, permute=None):
    """ObservationToArray: map characters to scalars ([B, rows, cols]) or vectors
    ([B, D, rows, cols]); raises RuntimeError on a character outside the mapping."""
    from pycolab_b200 import observers
    torch = _torch()
    table, valid, is_3d = observers.value_table(value_mapping, dtype)
    permute = observers.check_permute(permute, is_3d, 'ObservationToArray')
    unknown = torch.zeros((1,), dtype=torch.int32, device=self.device)
    out = observers.observe(self._lib, self._h, self._board, self.rows, self.cols, table,
                            valid, is_3d, permute, self._stream(), unknown)
    if int(unknown[0]):
      raise RuntimeError(
          'This ObservationToArray only knows array values for the characters {}, but it '
          'received an observation with a character not in that set'.format(
              ''.join(value_mapping.keys())))
    return out

  def repaint(self, character_mapping):
    """ObservationCharacterRepainter over every board: u8 [B, rows, cols]."""
    from pycolab_b200 import observers
    return observers.observe(self._lib, self._h, self._board, self.rows, self.cols,
                             observers.repaint_table(character_mapping), None, False, None,
                             self._stream())

  def sprite_state(self):
    """i32 [B, S, 8] device tensor of sprite records (PCL_S_* words)."""
    return self.sprites

  def frames(self):
    return self.plot[:, _lib.P_FRAME]

  def close(self):
    if getattr(self, '_h', None) is not None and self._h.value:
      self._lib.pcl_destroy(self._h)
      self._h = C.c_void_p()

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


def scrolling_crop_spec(rows, cols, sprite_index, pad_char=None, scroll_margins=(2, 3),
                        initial_offset=None, saccade=True, track=None):
  """Resolve ScrollingCropper constructor arguments (cropping.py:313-392).
  `track`: optional priority list replacing `sprite_index` — entries k > 0 mean
  sprite k - 1, k < 0 drape -k - 1 (`to_track` with several entities)."""
  if ((scroll_margins[0] is None and rows % 2 == 0) or
      (scroll_margins[1] is None and cols % 2 == 0)):
    raise ValueError("A ScrollingCropper can't perform perfectly-egocentric scrolling "
                     'with a window that has an even number of rows or columns. Either '
                     'specify looser scroll margins or use a window with odd dimensions.')
  m0 = rows // 2 if scroll_margins[0] is None else scroll_margins[0]
  m1 = cols // 2 if scroll_margins[1] is None else scroll_margins[1]
  if 2 * m0 >= rows or 2 * m1 >= cols:
    raise ValueError("A ScrollingCropper can't use scroll margins which extend to or "
                     'beyond the very centre of the scrolling window.')
  off = initial_offset if initial_offset is not None else (0, 0)
  spec = _lib.CropSpec(rows, cols, sprite_index, -1 if pad_char is None else ord(pad_char),
                       m0, m1, off[0], off[1], 1 if saccade else 0)
  if track is not None:
    if not 0 < len(track) <= _lib.MAX_TRACK or any(code == 0 for code in track):
      raise ValueError('a device cropper tracks 1..{} entities'.format(_lib.MAX_TRACK))
    for i, code in enumerate(track):
      spec.track[i] = int(code)
    spec.sprite_index = max(0, spec.track[0] - 1)
  return spec


def run_rotating(engines, actions, stream=None):
  """`len(actions)` steps from ONE C call (`pcl_run_many`): step t advances
  engines[t % len(engines)] with actions[t] (int32 device tensors).  No Python
  runs between the launches, so the call can sit inside a CUDA-graph capture."""
  torch = _torch()
  n, steps = len(engines), len(actions)
  handles = (C.c_void_p * n)(*[e._h.value for e in engines])
  outs = (C.c_void_p * n)(*[C.addressof(e._out) for e in engines])
  ptrs = (C.c_void_p * steps)()
  for t, a in enumerate(actions):
    e = engines[t % n]
    assert a.is_cuda and a.dtype == torch.int32 and a.is_contiguous()
    assert a.numel() == e.batch * e.actions_per_env
    if not e._showtime:
      raise RuntimeError('play() cannot be called until its_showtime() has been called')
    ptrs[t] = a.data_ptr()
  if stream is None:
    stream = engines[0]._stream()
  _lib.check(engines[0]._lib.pcl_run_many(handles, n, ptrs, outs, steps, stream),
             'pcl_run_many', engines[0]._h)
