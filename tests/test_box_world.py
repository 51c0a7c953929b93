"""Box-World (examples/research/box_world/box_world.py) on the device.

CPU: the set-up twin draws the original's levels, the oracle replays the original's
tapes, the tapes hold every event the rules distinguish, lowering accepts what the
kernel restates and refuses the rest.  GPU: the facade replays the tapes, and the
batched engine steps in lock-step with the oracle, with level rotation on auto-reset.
"""

import inspect
import json
import os
import sys

import numpy as np
import pytest

import box_world_cases as cases
import box_world_oracle as bo
import reference_trace as rt
from pycolab_b200 import _lib, lowering
from pycolab_b200.errors import NotLoweredError
from pycolab_b200.games import box_world as twin

gpu = pytest.mark.gpu


def _levels():
  with np.load(os.path.join(cases.GOLDEN_DIR, 'box_world_levels.npz')) as z:
    return {k: z[k] for k in z.files}


def _distractors(rows):
  return [(int(x), int(y)) for x, y in rows if x >= 0]


def _art_rows(art):
  return [bytes(row).decode('ascii') for row in art]


def _episodes(tape):
  """(art rows, distractors, frame indices) of every episode of a tape."""
  out = []
  for e in range(len(tape['art'])):
    frames = np.where(tape['episode'] == e)[0]
    out.append((_art_rows(tape['art'][e]), _distractors(tape['distractors'][e]), frames))
  return out


# ------------------------------------------------------------------ CPU: data

def test_twin_draws_the_original_levels():
  z = _levels()
  for name, params in cases.PARAMS.items():
    for i, seed in enumerate(z[name + '_seeds']):
      art, dist, player = twin.draw_level(*params, random_state=np.random.RandomState(int(seed)))
      assert art == _art_rows(z[name + '_art'][i]), (name, seed)
      assert dist == _distractors(z[name + '_distractors'][i]), (name, seed)
      assert tuple(player) == tuple(z[name + '_player'][i]), (name, seed)


def test_twin_keeps_the_generation_limit():
  # a room with space for two boxes at most: every attempt runs out of placements
  with pytest.raises(RuntimeError, match='MAX_GENERATION_TRIES'):
    twin.make_game(5, (4,), (4,), (0,), 1, random_state=np.random.RandomState(0))


@pytest.mark.parametrize('name', sorted(cases.TAPES))
def test_oracle_replays_the_original(name):
  tape = cases.load_tape(name)
  limit = int(tape['max_num_steps'])
  for art, dist, frames in _episodes(tape):
    world = bo.make_box_world(art, dist, limit)
    for t in frames:
      a = int(tape['action'][t])
      board, reward, discount = world.its_showtime() if tape['showtime'][t] else world.play(a)
      assert np.array_equal(board, tape['board'][t]), (name, t)
      assert (reward is not None) == bool(tape['has_reward'][t]), (name, t)
      if reward is not None:
        assert isinstance(reward, float) and reward == tape['reward'][t], (name, t)
      assert discount == tape['discount'][t] and world.game_over == bool(tape['game_over'][t])
      pl = world.things['.']
      assert (pl.row, pl.col, pl.aux['steps']) == tuple(tape['player'][t]), (name, t)
      assert np.array_equal(bo.box_world_plane(world) & 0x7f, tape['plane'][t]), (name, t)


def test_tapes_hold_every_event():
  seen = set()
  for name in cases.TAPES:
    seen |= cases.tape_events(cases.load_tape(name))
  assert cases.REQUIRED_EVENTS <= seen, cases.REQUIRED_EVENTS - seen


# -------------------------------------------------------------- CPU: lowering

def test_twin_lowers_like_the_original():
  with open(os.path.join(cases.GOLDEN_DIR, 'box_world_lowerings.json')) as f:
    want = json.load(f)
  for key, digest in want.items():
    seed = int(key.rsplit('_', 1)[1])
    game = twin.make_game(*cases.PARAMS['default'], random_state=np.random.RandomState(seed))
    assert rt.lowering_digest(lowering.lower(game)) == digest, key


def test_levels_share_one_signature():
  sigs = {lowering.lower(twin.make_game(*cases.PARAMS['default'],
                                        random_state=np.random.RandomState(s))).signature()
          for s in range(8)}
  assert len(sigs) == 1


def _spec_for(grid_size):
  game = twin.make_game(grid_size, (1,), (0,), (0,), 1, random_state=np.random.RandomState(1))
  return lowering.lower(game).make_spec(True)


def _create(spec):
  import ctypes as C
  lib = _lib.load()
  h = C.c_void_p()
  status = lib.pcl_create(C.byref(spec), 4, -1, C.byref(h))
  if status == _lib.OK:
    lib.pcl_destroy(h)
  return status


def test_pcl_create_board_limits():
  assert _create(_spec_for(12)) == _lib.OK           # 14 x 14
  assert _create(_spec_for(30)) == _lib.OK           # 32 x 32
  spec = _spec_for(30)
  spec.rows = spec.cols = 33
  spec.pitch, spec.bits_words = 48, 12
  assert _create(spec) == _lib.ERR_UNSUPPORTED
  spec = _spec_for(12)
  spec.program_arg[1], spec.program_arg[2] = 4, 0    # rotation over no levels
  assert _create(spec) == _lib.ERR_INVALID


def test_grid_size_31_is_refused():
  game = twin.make_game(31, (1,), (0,), (0,), 1, random_state=np.random.RandomState(0))
  with pytest.raises(NotLoweredError, match='32 x 32'):
    lowering.lower(game)


def _level_engine(schedule=None, z_order=None):
  from pycolab_b200 import ascii_art
  art, dist, (x, y) = twin.draw_level(*cases.PARAMS['default'],
                                      random_state=np.random.RandomState(3))
  chars = sorted(set(''.join(art)) - set(' #.'))
  grid = np.array([list(r) for r in art])
  drapes = {}
  for ch in chars:
    klass = twin.GemDrape if ch == '*' else twin.KeyDrape if ch.islower() else twin.LockDrape
    ys, xs = np.where(grid == ch)
    drapes[ch] = ascii_art.Partial(klass, x=int(xs[-1]), y=int(ys[-1]))
  sprites = {'.': ascii_art.Partial(twin.PlayerSprite, 12, x, y, dist, 120)}
  return ascii_art.ascii_art_to_game(
      art, ' ', sprites=sprites, drapes=drapes,
      update_schedule=schedule(chars) if schedule else ['.'] + chars,
      z_order=z_order(chars) if z_order else chars + ['.'])


def test_schedule_and_z_order_are_checked():
  lowering.lower(_level_engine())
  with pytest.raises(NotLoweredError, match='update group'):
    lowering.lower(_level_engine(schedule=lambda c: [['.'], c]))
  with pytest.raises(NotLoweredError, match='update group'):
    lowering.lower(_level_engine(schedule=lambda c: c[::-1] + ['.']))
  with pytest.raises(NotLoweredError, match='z_order'):
    lowering.lower(_level_engine(z_order=lambda c: ['.'] + c))


@pytest.fixture
def compat_loader(tmp_path):
  """Writes a module source into tmp_path and loads it through `compat`, the way a
  user's copy of the example file is loaded."""
  from pycolab_b200 import compat
  saved = {k: v for k, v in sys.modules.items() if k == 'pycolab' or k.startswith('pycolab.')}
  compat.uninstall()
  compat.install()

  def load(source, copy):
    path = tmp_path / copy / 'box_world.py'
    path.parent.mkdir(exist_ok=True)
    path.write_text(source)
    return compat.load_example(str(path))
  yield load
  compat.uninstall()
  sys.modules.update(saved)


def test_edited_copies_are_refused(compat_loader, monkeypatch):
  """A user's copy of the set-up lowers while its classes are token-for-token the
  known ones (pointed here at the copy's own classes) and its module constants are
  the original's; an edited update(), an edited BoxThing or an edited REWARD_GOAL is
  refused, never replaced by the stock kernel."""
  from pycolab_b200 import _fingerprints
  src = inspect.getsource(twin).replace('from pycolab_b200 import', 'from pycolab import') \
      .replace('from pycolab_b200.prefab_parts', 'from pycolab.prefab_parts')
  mod = compat_loader(src, 'plain')
  for name in ('PlayerSprite', 'GemDrape', 'KeyDrape', 'LockDrape', 'BoxThing'):
    monkeypatch.setitem(_fingerprints.KNOWN, ('box_world', name),
                        lowering.source_fingerprint(inspect.getsource(getattr(mod, name))))
  make = lambda m: m.make_game(*cases.PARAMS['default'], random_state=np.random.RandomState(0))
  rt_digest = rt.lowering_digest(lowering.lower(make(mod)))
  assert rt_digest == rt.lowering_digest(lowering.lower(make(twin)))
  gem_update = "    raise NotImplementedError('runs on the device: csrc/box_world.cu')\n\n\nclass KeyDrape"
  assert gem_update in src
  edits = {
      'update': src.replace(gem_update, "    the_plot.add_reward(5.)\n\n\nclass KeyDrape"),
      'base': src.replace('    self.curtain[y][x] = True', '    self.curtain[y][x] = False'),
      'constant': src.replace('REWARD_GOAL = 10.', 'REWARD_GOAL = 11.'),
  }
  for copy, edited in edits.items():
    assert edited != src, copy
    with pytest.raises(NotLoweredError, match='differs'):
      lowering.lower(make(compat_loader(edited, copy)))


def test_cycle_levels_is_refused_where_it_does_not_apply():
  from pycolab_b200 import batched, levels
  from pycolab_b200.games import shockwave
  pool = [twin.make_game(*cases.PARAMS['default'], random_state=np.random.RandomState(s))
          for s in range(2)]
  with pytest.raises(ValueError, match='box_world'):
    batched.BatchedEngine([shockwave.make_game(levels.shockwave_level(s)) for s in range(2)],
                          batch=4, cycle_levels=True)
  with pytest.raises(ValueError, match='more than one level'):
    batched.BatchedEngine(pool[:1], batch=4, cycle_levels=True)
  with pytest.raises(ValueError, match='share_levels'):
    batched.BatchedEngine(pool, batch=4, cycle_levels=True, share_levels=False)


# ------------------------------------------------------------------------ GPU

@gpu
@pytest.mark.parametrize('name', sorted(cases.TAPES))
def test_facade_replays_the_original(name):
  """The Engine facade (B = 1) on every episode of a tape: boards, float rewards,
  discounts, every drape's curtain and the player after every frame."""
  tape = cases.load_tape(name)
  limit = int(tape['max_num_steps'])
  for art, dist, frames in _episodes(tape):
    game = twin.game_from_art(art, dist, limit)
    drapes = [ch for ch in game.things if ch != '.']
    for t in frames:
      obs, reward, discount = (game.its_showtime() if tape['showtime'][t]
                               else game.play(int(tape['action'][t])))
      assert np.array_equal(obs.board, tape['board'][t]), (name, t)
      if tape['has_reward'][t]:
        assert type(reward) is float and reward == tape['reward'][t], (name, t, reward)
      else:
        assert reward is None, (name, t)
      assert discount == tape['discount'][t] and game.game_over == bool(tape['game_over'][t])
      pl = game.things['.']
      assert (pl.position[0], pl.position[1], pl._step_counter) == tuple(tape['player'][t])
      for ch in drapes:
        assert np.array_equal(game.things[ch].curtain, tape['plane'][t] == ord(ch)), (name, t, ch)


def _pool(n, params='default', seed0=0, limit=120):
  levels = []
  for s in range(seed0, seed0 + n):
    art, dist, _ = twin.draw_level(*cases.PARAMS[params] if isinstance(params, str) else params,
                                   random_state=np.random.RandomState(s))
    levels.append((art, dist, limit))
  return levels


def _check(eng, worlds, outs, t, envs=None):
  import torch
  torch.cuda.synchronize()
  envs = range(eng.batch) if envs is None else envs
  boards = eng.board.cpu().numpy()
  plane = eng.plane()[:, :, :eng.cols].cpu().numpy()
  reward, has = eng.reward.cpu().numpy(), eng.has_reward.cpu().numpy()
  disc, done = eng.discount.cpu().numpy(), eng.done.cpu().numpy()
  for k, e in enumerate(envs):
    board, r, d = outs[k]
    w = worlds[k]
    assert np.array_equal(boards[e], board), (t, e)
    assert np.array_equal(plane[e], bo.box_world_plane(w)), (t, e)
    assert bool(has[e]) == (r is not None), (t, e)
    assert int(reward[e]) == (0 if r is None else r), (t, e)
    assert float(disc[e]) == d and bool(done[e]) == w.game_over, (t, e)


def _lockstep(B, levels, steps, policy, cycle, auto_reset=True, resets=(), seed=0):
  """BatchedEngine vs one oracle world per env, every env checked every step."""
  import torch
  from pycolab_b200 import batched
  n = len(levels)
  games = [twin.game_from_art(*lvl) for lvl in levels]
  eng = batched.BatchedEngine(games, batch=B, auto_reset=auto_reset, cycle_levels=cycle)
  lvl = eng.level.cpu().numpy().copy()
  assert np.array_equal(lvl, np.arange(B) % n)
  worlds = [bo.make_box_world(*levels[lvl[e]]) for e in range(B)]
  outs = [w.its_showtime() for w in worlds]
  eng.its_showtime()
  _check(eng, worlds, outs, -1)
  rng = np.random.RandomState(seed)
  restarts = 0
  for t in range(steps):
    if t in resets:                                  # masked reset keeps the level
      mask = rng.rand(B) < 0.3
      eng.reset(torch.from_numpy(mask.astype(np.uint8)).cuda())
      assert np.array_equal(eng.level.cpu().numpy(), lvl)
      for e in np.where(mask)[0]:
        worlds[e] = bo.make_box_world(*levels[lvl[e]])
        outs[e] = worlds[e].its_showtime()
      _check(eng, worlds, outs, t)
    actions = np.array([cases.policy_action(outs[e][0], rng, policy, 0.2) for e in range(B)],
                       dtype=np.int32)
    eng.play(torch.from_numpy(actions).cuda())
    new_lvl = eng.level.cpu().numpy()
    for e in range(B):
      if worlds[e].game_over:
        if not auto_reset:
          continue                                   # frozen: outputs stay as they were
        want = (lvl[e] + B) % n if cycle else lvl[e]
        assert new_lvl[e] == want, (t, e)
        worlds[e] = bo.make_box_world(*levels[new_lvl[e]])
        outs[e] = worlds[e].its_showtime()
        restarts += 1
      else:
        assert new_lvl[e] == lvl[e]
        outs[e] = worlds[e].play(int(actions[e]))
    lvl = new_lvl.copy()
    _check(eng, worlds, outs, t)
  assert not eng.error_codes().any()
  return restarts


@gpu
@pytest.mark.parametrize('cycle', [False, True])
@pytest.mark.parametrize('policy', ['scripted', 'random'])
def test_batched_lockstep_13(cycle, policy):
  # a 40-move limit: random walks end by timeout too, so every env changes level
  restarts = _lockstep(13, _pool(48, limit=40), 300, policy, cycle, resets=(40, 150))
  assert restarts >= 13


@gpu
def test_batched_lockstep_4097_cycling():
  levels = _pool(24) + _pool(24, 'backward', 700)
  assert _lockstep(4097, levels, 40, 'random', True, resets=(20,)) > 0


@gpu
def test_batched_large_boards():
  # 22 x 22 and 32 x 32 rooms: two 16-byte segments per lane
  _lockstep(37, _pool(48, 'large', 900), 120, 'scripted', True)
  _lockstep(9, _pool(8, (30, (1, 2, 3, 4), (0, 1, 2, 3, 4), (0,), 1), 950), 150, 'scripted', True)


@gpu
def test_frozen_without_auto_reset():
  _lockstep(13, _pool(48, 'default', 300, limit=20), 60, 'random', False, auto_reset=False)


@gpu
def test_shards_reproduce_one_engine():
  import torch
  from pycolab_b200 import batched, dist
  levels = _pool(48, 'default', 1200, limit=25)
  B = 21
  one = batched.BatchedEngine([twin.game_from_art(*l) for l in levels], batch=B,
                              cycle_levels=True)
  shards = [dist.make_shard_engine([twin.game_from_art(*l) for l in levels], B, r, 2, 0,
                                   cycle_levels=True) for r in range(2)]
  outs = [one.its_showtime()] + [s.its_showtime() for s in shards]
  rng = np.random.RandomState(5)
  for t in range(200):
    a = torch.from_numpy(rng.choice([0, 1, 2, 3, -1], size=B).astype(np.int32)).cuda()
    one.play(a)
    shards[0].play(a[:shards[0].batch].contiguous())
    shards[1].play(a[shards[0].batch:].contiguous())
    torch.cuda.synchronize()
    for name in ('board', 'reward', 'has_reward', 'discount', 'done', 'level'):
      whole = getattr(one, name)
      parts = torch.cat([getattr(s, name) for s in shards])
      assert torch.equal(whole, parts), (t, name)
  assert not torch.equal(one.level, torch.arange(B, device=one.level.device).int() % 48)


@gpu
def test_sampled_envs_at_scale():
  """16 384 envs over a pool of 1024 levels for 500 steps with device-drawn actions;
  64 sampled envs replayed on the oracle, level changes taken from eng.level."""
  import torch
  from pycolab_b200 import batched
  levels = _pool(1024, 'default', 20000)
  B, T = 16384, 500
  eng = batched.BatchedEngine([twin.game_from_art(*l) for l in levels], batch=B,
                              cycle_levels=True)
  sample = np.random.RandomState(1).choice(B, 64, replace=False)
  idx = torch.from_numpy(sample).cuda()
  lvl = eng.level.cpu().numpy()[sample]
  worlds = [bo.make_box_world(*levels[l]) for l in lvl]
  outs = [w.its_showtime() for w in worlds]
  eng.its_showtime()
  _check(eng, worlds, outs, -1, envs=sample)
  table = torch.tensor([0, 1, 2, 3, 0, 1, 2, 3, -1, 4], dtype=torch.int32, device='cuda')
  gen = torch.Generator(device='cuda')
  gen.manual_seed(3)
  for t in range(T):
    a = table[torch.randint(0, len(table), (B,), device='cuda', generator=gen)]
    eng.play(a)
    acts = a[idx].cpu().numpy()
    new_lvl = eng.level[idx].cpu().numpy()
    for k in range(len(sample)):
      if worlds[k].game_over:
        assert new_lvl[k] == (lvl[k] + B) % len(levels)
        worlds[k] = bo.make_box_world(*levels[new_lvl[k]])
        outs[k] = worlds[k].its_showtime()
      else:
        outs[k] = worlds[k].play(int(acts[k]))
    lvl = new_lvl
    _check(eng, worlds, outs, t, envs=sample)
  assert not eng.error_codes().any()


@gpu
def test_original_file_through_compat_if_present():
  """The original's box_world.py, loaded through compat, lowers and steps."""
  import refdriver
  if not refdriver.available():
    pytest.skip(refdriver.MISSING)
  from pycolab_b200 import compat
  path = os.path.join(refdriver.REFERENCE_ROOT, 'pycolab', 'examples', 'research', 'box_world',
                      'box_world.py')
  module = compat.load_example(path)
  game = module.make_game(*cases.PARAMS['default'], random_state=np.random.RandomState(0))
  obs, reward, discount = game.its_showtime()
  assert reward is None and discount == 1.0
  obs, reward, discount = game.play(0)
  assert reward == 0.0 and type(reward) is float
