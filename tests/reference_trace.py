"""Seeded scenarios that pin the oracle (`oracle/`) to the original pycolab.

Each scenario plays one game on one kind of engine (a `side`) and folds every
value the comparison looks at (boards, rewards, discounts, game-over flags,
sprite registers, curtains, crops, ...) into a `Trace`: a CRC-32 chained over
the records, kept every `Trace.EVERY` records and at the end.  The original
pycolab's traces are stored in `tests/golden/reference_traces.npz`
(`tests/golden/make_reference_traces.py` writes them from an upstream pycolab
checkout); `tests/test_oracle_vs_reference.py` replays the same scenarios on the
oracle and compares the two traces checkpoint by checkpoint.

A side provides the constructors and the few accessors that differ between an
original pycolab Engine and an oracle World: `OracleSide` here,
`refdriver.ReferenceSide` for the original.
"""

import contextlib
import random
import struct
import zlib

import numpy as np

from oracle import engine_model as em
from oracle import games
from pycolab_b200 import levels
import golden_cases as gc


class Trace(object):
  """Chained CRC-32 of a sequence of records (one or more per frame)."""
  EVERY = 16

  def __init__(self):
    self.crc = 0
    self.records = 0
    self.marks = []

  def add(self, *parts):
    for p in parts:
      self.crc = zlib.crc32(_canon(p), self.crc)
    self.records += 1
    if self.records % self.EVERY == 0:
      self.marks.append(self.crc)

  def result(self):
    return np.array(self.marks + [self.crc, self.records], dtype=np.uint32)


def _canon(x):
  """Bytes of a value that do not depend on which engine produced it: arrays by
  shape and element values (not dtype), numbers by value, the rest by repr."""
  if isinstance(x, np.ndarray):
    return repr(x.shape).encode() + np.ascontiguousarray(x, dtype=np.int64).tobytes()
  if isinstance(x, (bool, np.bool_)):
    return b'T' if x else b'F'
  if isinstance(x, (int, np.integer)):
    return struct.pack('<q', int(x))
  if isinstance(x, (float, np.floating)):
    return struct.pack('<d', float(x))
  if isinstance(x, (tuple, list)):
    return b'(' + b','.join(_canon(v) for v in x) + b')'
  if isinstance(x, dict):
    return _canon(sorted(x.items()))
  return repr(x).encode()


def lowering_digest(game):
  """CRC-32 of everything a lowered game (`lowering.LoweredGame`) hands the device."""
  trace = Trace()
  trace.add(game.signature(), game.backdrop, game.sprites, game.drapes, game.plot,
            game.patterns, game.bits, game.drape_kind, game.dynamic_z,
            game.reward_type.__name__, game.backdrop_role)
  return trace.crc


@contextlib.contextmanager
def sorted_default_schedule():
  """Without an update_schedule, ascii_art_to_game updates the entities in set
  order, like the original (ascii_art.py:161), and that order follows the string
  hash seed of the process.  A stored lowering needs one order: the sorted one."""
  from pycolab_b200 import ascii_art
  build = ascii_art.ascii_art_to_game

  def sorted_build(art, what_lies_beneath, sprites=None, drapes=None, *args, **kwargs):
    if len(args) < 2 and kwargs.get('update_schedule') is None:
      kwargs['update_schedule'] = sorted(set(sprites or {}) | set(drapes or {}))
    return build(art, what_lies_beneath, sprites, drapes, *args, **kwargs)
  ascii_art.ascii_art_to_game = sorted_build
  try:
    yield
  finally:
    ascii_art.ascii_art_to_game = build


def check_lowering(key, game):
  """`game` lowers exactly like the original's example of the same name did
  (tests/golden/reference_lowerings.json)."""
  import json
  import os
  path = os.path.join(gc.GOLDEN_DIR, 'reference_lowerings.json')
  with open(path) as f:
    want = json.load(f)[key]
  assert lowering_digest(game) == want, '%s lowers unlike the original' % key


def board_of(out):
  return np.asarray(getattr(out[0], 'board', out[0]))


def sprites_of(engine):
  """{char: (row, col, visible)} of every sprite (things with a position)."""
  out = {}
  for ch, ent in engine.things.items():
    if hasattr(ent, 'position'):
      out[ch] = (int(ent.position[0]), int(ent.position[1]), bool(ent.visible))
  return out


def reward_pair(reward):
  return (0, 0) if reward is None else (int(reward), 1)


def frame(trace, engine, out, sprites=True):
  """The frame compared by every lock-step scenario."""
  trace.add(board_of(out), reward_pair(out[1]), float(out[2]), bool(engine.game_over))
  if sprites:
    trace.add(sprites_of(engine))


class OracleSide(object):
  """The oracle restatement, on the art the original's stock levels use."""

  def scrolly_stock(self, level):
    maze, board, beneath = gc.scrolly_art(gc.load('scrolly_stock_L%d' % level))
    return lambda: games.make_scrolly_maze(maze, board, '+', beneath)

  def scrolly(self, maze, board, beneath):
    return lambda: games.make_scrolly_maze(maze, board, '+', beneath)

  def warehouse_stock(self, level):
    art, wlb = gc.warehouse_art(gc.load('warehouse_stock_L%d' % level))
    return lambda: games.make_warehouse(art, wlb)

  def warehouse(self, art, beneath):
    return lambda: games.make_warehouse(art, beneath)

  def marauders(self, seed):
    rng = np.random.RandomState(seed)     # one stream across episodes
    art = levels.marauders_level()
    return lambda: games.make_marauders(art, rng)

  def fixture(self, art, walkers, scrollys=None, **kw):
    return games.make_fixture_world(art, ' ', walkers, scrollys, **kw)

  def fixture_action(self, action):
    return action

  def walk_result(self, engine, ch):
    return engine.things[ch].last_result

  def classic(self, kind, art):
    import importlib
    art = art or list(importlib.import_module('pycolab_b200.games.classics.' + kind).GAME_ART)
    return lambda: games.make_classic(kind, art)

  def aperture(self, level, art):
    if art is None:
      art = [bytes(r).decode('ascii') for r in gc.load('aperture_stock_L%d' % level)['art']]
    return lambda: games.make_aperture(art)

  def fluvial(self, art):
    from pycolab_b200.games import fluvial_natation
    art = art or list(fluvial_natation.GAME_ART)
    return lambda: games.make_fluvial(art)

  def scrolly_cropper(self, engine, pad, margins):
    crop = em.ScrollingCrop(9, 9, ['P'], pad_char=pad, scroll_margins=margins)
    crop.set_engine(engine)
    return lambda out: crop.crop(out[0])

  def ordeal(self):
    from test_ordeal import OracleOrdeal
    return OracleOrdeal()

  def ordeal_chapter(self, story):
    return story.chapter

  def apprehend(self, seed):
    from pycolab_b200.games import apprehend
    return games.make_apprehend(list(apprehend.GAME_ART), random.Random(seed))

  def ball_registers(self, engine):
    aux = engine.things['b'].aux
    return float(aux['dx']), float(aux['acc'])

  def shockwave(self, level, seed):
    return games.make_shockwave(level, np.random.RandomState(seed))

  def shockwave_stock_art(self):
    from pycolab_b200.games import shockwave
    return shockwave.LEVELS[0]


ORACLE = OracleSide()


# ------------------------------------------------------------------ scenarios
# Each returns (trace, facts): facts are counts the test asserts on besides the
# trace (episodes played, shots fired, ...).

def lockstep(make, actions, sprites=True, per_frame=None):
  """Step with auto-reset on game over, recording every frame."""
  trace = Trace()
  env = make()
  out = env.its_showtime()
  episodes = 0
  for a in actions:
    frame(trace, env, out, sprites)
    if per_frame is not None:
      per_frame(trace, env, out)
    if env.game_over:
      episodes += 1
      env = make()
      out = env.its_showtime()
      continue
    out = env.play(a)
  return trace, dict(episodes=episodes)


def scrolly_stock(side, level):
  actions = np.random.RandomState(100 + level).randint(0, 5, size=1500).tolist()
  return lockstep(side.scrolly_stock(level), actions)


def scrolly_stock_with_quit(side):
  actions = np.random.RandomState(7).randint(0, 6, size=400).tolist()
  return lockstep(side.scrolly_stock(0), actions)


def scrolly_generated_64(side, seed):
  maze, board, beneath = levels.scrolly_maze_level(seed)
  rs = np.random.RandomState(seed)
  # biased walk so the window actually scrolls a lot
  actions = rs.choice([0, 1, 2, 3, 4], size=600, p=[.3, .15, .3, .15, .1]).tolist()
  return lockstep(side.scrolly(maze, board, beneath), actions)


def warehouse_stock(side, level):
  actions = np.random.RandomState(200 + level).randint(0, 5, size=1500).tolist()
  return lockstep(side.warehouse_stock(level), actions)


def warehouse_generated_80(side):
  art = levels.warehouse_level(3)
  actions = np.random.RandomState(3).randint(0, 4, size=800).tolist()
  return lockstep(side.warehouse(art, ' '), actions)


def marauders_stock(side, seed):
  actions = np.random.RandomState(300 + seed).randint(0, 4, size=1200).tolist()
  return lockstep(side.marauders(seed), actions)


def _random_fixture_case(seed):
  rs = np.random.RandomState(seed)
  H, W = int(rs.randint(5, 12)), int(rs.randint(5, 14))
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[rs.random_sample((H, W)) < 0.25] = ord('#')
  art[rs.random_sample((H, W)) < 0.1] = ord('%')
  free = np.argwhere(art == ord(' '))
  picks = free[rs.permutation(len(free))[:3]]
  for ch, (r, c) in zip('abc', picks):
    art[r, c] = ord(ch)
  walkers = {
      'a': dict(impassable='#', confined=bool(rs.randint(2))),
      'b': dict(impassable='#%a', confined=bool(rs.randint(2))),
      'c': dict(impassable='', confined=False),
  }
  schedule = [['a'], ['b', 'c']] if rs.randint(2) else [['a', 'b', 'c']]
  art = [bytes(r).decode('ascii') for r in art]
  return art, walkers, schedule, rs


def fixture_walkers_random(side, seed):
  """MazeWalkers on random art: every frame, then each walker's motion result
  and virtual position after every step."""
  art, walkers, schedule, rs = _random_fixture_case(seed)
  stream = [{ch: int(rs.randint(0, 9)) for ch in 'abc'} for _ in range(300)]
  env = side.fixture(art, walkers, update_schedule=schedule, z_order='abc')
  out = env.its_showtime()
  trace = Trace()
  for act in stream:
    frame(trace, env, out)
    out = env.play(side.fixture_action(act))
    trace.add([(side.walk_result(env, ch), tuple(env.things[ch].virtual_position))
               for ch in 'abc'])
  return trace, {}


def fixture_scrolly_random(side, seed, margins):
  """A Scrolly and two walkers in one scrolling group; the curtain after every
  step.  The original raises when a no-margin Scrolly clips a diagonal order to
  (0, 0) (sprites.py:449-454): the frame where that happens ends the trace."""
  rs = np.random.RandomState(1000 + seed)
  PH, PW, H, W = 17, 23, 8, 11
  pattern = rs.random_sample((PH, PW)) < 0.2
  corner = (int(rs.randint(0, PH - H + 1)), int(rs.randint(0, PW - W + 1)))
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[3, 4] = ord('P')
  art[5, 7] = ord('q')
  art = [bytes(r).decode('ascii') for r in art]
  walkers = {'P': dict(impassable='#', egocentric=True),
             'q': dict(impassable='#', egocentric=bool(seed % 2))}
  scrollys = {'#': dict(pattern=pattern, corner=corner, margins=margins)}
  env = side.fixture(art, walkers, scrollys, update_schedule=[['#'], ['P', 'q']],
                     z_order='#Pq')
  out = env.its_showtime()
  trace = Trace()
  for t in range(400):
    frame(trace, env, out)
    m = int(rs.randint(0, 9))         # everybody in the group requests the same motion
    try:
      out = env.play(side.fixture_action(m))
    except RuntimeError:
      trace.add('raised')
      return trace, dict(raised_at=t)
    trace.add(env.things['#'].curtain)
  return trace, dict(raised_at=None)


def classics(side, kind, art):
  art = None if art == 'stock' else levels.classic_level(kind)
  n_actions = 3 if kind == 'chain_walk' else 6     # includes no-op / unmapped actions
  actions = np.random.RandomState(len(kind)).randint(0, n_actions, size=2500).tolist()
  rewards = []

  def reward_type(trace, env, out):   # float rewards: the type is compared too
    trace.add(type(out[1]).__name__)
    rewards.append(out[1])
  trace, facts = lockstep(side.classic(kind, art), actions, per_frame=reward_type)
  facts['rewards'] = sum(r is not None for r in rewards)
  return trace, facts


def aperture_actions(seed, n):
  """Walks, blaster shots in all directions, idle steps and a rare quit."""
  rs = np.random.RandomState(seed)
  return rs.choice(list(range(10)), size=n,
                   p=[.14, .14, .14, .14, .04, .1, .1, .1, .095, .005]).tolist()


def aperture(side, level):
  if level == 'other':
    make, seed = side.aperture(None, levels.aperture_level()), 43
  else:
    make, seed = side.aperture(level, None), 40 + level
  shots = []

  def curtain(trace, env, out):
    trace.add(env.things['X'].curtain)
    shots.append(int(np.asarray(env.things['X'].curtain).sum() > 0))
  trace, facts = lockstep(make, aperture_actions(seed, 3000), per_frame=curtain)
  facts['shots'] = sum(shots)
  return trace, facts


def fluvial_natation(side, art):
  art = None if art == 'stock' else levels.fluvial_level()
  actions = np.random.RandomState(5).choice([0, 1, 2], size=1500, p=[.2, .6, .2]).tolist()
  return lockstep(side.fluvial(art), actions)


def scrolling_cropper(side, pad, margins):
  """ScrollingCropper 9x9 tracking 'P' over a generated 32x32 scrolly_maze."""
  maze, board, beneath = levels.scrolly_maze_level(5, world_shape=(65, 65),
                                                   board_shape=(32, 32))
  env = side.scrolly(maze, board, beneath)()
  crop = side.scrolly_cropper(env, pad, margins)
  out = env.its_showtime()
  rs = np.random.RandomState(11)
  trace = Trace()
  for _ in range(300):
    trace.add(np.asarray(crop(out)))
    if env.game_over:
      break
    a = int(rs.randint(0, 5))
    out = env.play(a)
  return trace, {}


def ordeal_story(side, seed):
  """examples/ordeal.py's Story: after every step the chapter, the (cropped in
  kansas) board, the summed reward, the discount and game over."""
  rs = np.random.RandomState(500 + seed)
  story = side.ordeal()
  story.its_showtime()
  trace = Trace()
  for a in rs.choice([0, 1, 2, 3], size=700, p=[.3, .2, .2, .3]).tolist():
    if story.game_over:
      break
    out = story.play(a)
    trace.add(side.ordeal_chapter(story), board_of(out),
              None if out[1] is None else float(out[1]), float(out[2]), bool(story.game_over))
  return trace, {}


def apprehend_many_episodes(side):
  """examples/apprehend.py, 200 seeded episodes: boards, rewards (value and type),
  discounts and the ball's float64 registers."""
  trace = Trace()
  steps = wins = 0
  for seed in range(200):
    env = side.apprehend(seed)
    out = env.its_showtime()
    rs = np.random.RandomState(seed)
    while True:
      trace.add(board_of(out), repr(out[1]), type(out[1]).__name__, float(out[2]),
                bool(env.game_over), side.ball_registers(env))
      if env.game_over:
        wins += out[1] == 1
        break
      out = env.play(int(rs.randint(0, 3)))
      steps += 1
  return trace, dict(steps=steps, wins=wins)


def shockwave_many_episodes(side, level):
  """examples/shockwave.py (scipy's distance transform, NumPy's randint): boards,
  rewards, discounts and the wave's curtain every step of 80 seeded episodes."""
  art = side.shockwave_stock_art() if level == 'stock' else levels.shockwave_level(7, 14, 31, 0.5)
  trace = Trace()
  steps = ends = 0
  for seed in range(80):
    env = side.shockwave(art, seed)
    out = env.its_showtime()
    rs = np.random.RandomState(100 + seed)
    for _ in range(300):
      trace.add(board_of(out), env.things['@'].curtain, repr(out[1]), type(out[1]).__name__,
                float(out[2]), bool(env.game_over))
      if env.game_over:
        ends += 1
        break
      out = env.play(int(rs.choice([0, 1, 2, 3, 4], p=[.55, .15, .15, .1, .05])))
      steps += 1
  return trace, dict(steps=steps, ends=ends)


def cases():
  """{golden key: (scenario, args)} of every stored trace."""
  out = {}
  for level in (0, 1, 2):
    out['scrolly_stock_%d' % level] = (scrolly_stock, (level,))
    out['warehouse_stock_%d' % level] = (warehouse_stock, (level,))
    out['aperture_%d' % level] = (aperture, (level,))
  out['aperture_other'] = (aperture, ('other',))
  out['scrolly_stock_with_quit'] = (scrolly_stock_with_quit, ())
  for seed in (0, 1):
    out['scrolly_generated_64_%d' % seed] = (scrolly_generated_64, (seed,))
  out['warehouse_generated_80'] = (warehouse_generated_80, ())
  for seed in (0, 1, 2):
    out['marauders_stock_%d' % seed] = (marauders_stock, (seed,))
  for seed in range(8):
    out['fixture_walkers_%d' % seed] = (fixture_walkers_random, (seed,))
  for seed, margins in FIXTURE_SCROLLY:
    out['fixture_scrolly_%d' % seed] = (fixture_scrolly_random, (seed, margins))
  for kind in games.CLASSIC_KINDS:
    for art in ('stock', 'other'):
      out['classic_%s_%s' % (kind, art)] = (classics, (kind, art))
  for art in ('stock', 'other'):
    out['fluvial_%s' % art] = (fluvial_natation, (art,))
  for i, (pad, margins) in enumerate(CROPPERS):
    out['cropper_%d' % i] = (scrolling_cropper, (pad, margins))
  for seed in range(6):
    out['ordeal_%d' % seed] = (ordeal_story, (seed,))
  out['apprehend'] = (apprehend_many_episodes, ())
  for level in ('stock', 'generated'):
    out['shockwave_%s' % level] = (shockwave_many_episodes, (level,))
  return out


FIXTURE_SCROLLY = [(0, (2, 3)), (1, None), (2, (1, 1)), (3, None), (4, (2, 2)), (5, (1, 2))]
CROPPERS = [(' ', (None, None)), (None, (2, 3)), (' ', (2, 3))]
