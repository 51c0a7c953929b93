"""Drive the original pycolab (an upstream checkout) on arbitrary art.

Set PYCOLAB_UPSTREAM to the directory that holds the upstream `pycolab` package.
The generators under `tests/golden/` use it to produce the committed golden
fixtures; the one test that runs an upstream example file itself on the device
skips without it.  Nothing else in the suite needs it.
"""

import os
import sys

import numpy as np

REFERENCE_ROOT = os.environ.get('PYCOLAB_UPSTREAM', '')
MISSING = 'needs an upstream pycolab checkout (set PYCOLAB_UPSTREAM)'


def available():
  return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, 'pycolab'))


def _import():
  if REFERENCE_ROOT not in sys.path:
    sys.path.insert(0, REFERENCE_ROOT)
  import warnings
  warnings.filterwarnings('ignore', category=DeprecationWarning)
  from pycolab import ascii_art, cropping
  from pycolab.examples import (scrolly_maze, warehouse_manager,
                                extraterrestrial_marauders)
  from pycolab.tests import test_things
  return dict(ascii_art=ascii_art, cropping=cropping, scrolly_maze=scrolly_maze,
              warehouse_manager=warehouse_manager,
              extraterrestrial_marauders=extraterrestrial_marauders,
              test_things=test_things)


def ref_scrolly_maze(maze_art, board_art, beneath='#', level=None):
  m = _import()['scrolly_maze']
  if level is not None:
    return m.make_game(level)
  saved = (m.MAZES_ART, m.MAZES_WHAT_LIES_BENEATH, m.STAR_ART)
  try:
    m.MAZES_ART = [maze_art]
    m.MAZES_WHAT_LIES_BENEATH = [beneath]
    m.STAR_ART = board_art
    return m.make_game(0)
  finally:
    m.MAZES_ART, m.MAZES_WHAT_LIES_BENEATH, m.STAR_ART = saved


def ref_stock_scrolly_art(level):
  m = _import()['scrolly_maze']
  return (list(m.MAZES_ART[level]), list(m.STAR_ART),
          m.MAZES_WHAT_LIES_BENEATH[level])


def ref_better_scrolly(art=None, level=None):
  sys.path.insert(0, REFERENCE_ROOT) if REFERENCE_ROOT not in sys.path else None
  _import()
  from pycolab.examples import better_scrolly_maze as m
  if level is not None:
    return m.make_game(level)
  saved = m.MAZES_ART
  try:
    m.MAZES_ART = [art]
    return m.make_game(0)
  finally:
    m.MAZES_ART = saved


def ref_better_scrolly_stock(level):
  """(art, STARTER_OFFSET, TEASER_CORNER) of a stock better_scrolly_maze level."""
  _import()
  from pycolab.examples import better_scrolly_maze as m
  return list(m.MAZES_ART[level]), tuple(m.STARTER_OFFSET[level]), tuple(m.TEASER_CORNER[level])


def ref_better_scrolly_croppers(level):
  _import()
  from pycolab.examples import better_scrolly_maze as m
  return m.make_croppers(level)


def ref_classic(kind, art=None):
  """examples/classics/{four_rooms,cliff_walk,chain_walk}.make_game, optionally
  on other art."""
  _import()
  import importlib
  m = importlib.import_module('pycolab.examples.classics.' + kind)
  if art is None:
    return m.make_game()
  saved = m.GAME_ART
  try:
    m.GAME_ART = art
    return m.make_game()
  finally:
    m.GAME_ART = saved


def ref_classic_art(kind):
  _import()
  import importlib
  return list(importlib.import_module('pycolab.examples.classics.' + kind).GAME_ART)


def ref_fluvial(art=None):
  _import()
  from pycolab.examples import fluvial_natation as m
  if art is None:
    return m.make_game()
  saved = m.GAME_ART
  try:
    m.GAME_ART = art
    return m.make_game()
  finally:
    m.GAME_ART = saved


def ref_fluvial_art():
  _import()
  from pycolab.examples import fluvial_natation as m
  return list(m.GAME_ART)


def ref_aperture(level=None, art=None):
  _import()
  from pycolab.examples import aperture as m
  if art is None:
    return m.make_game(level)
  saved = m.LEVELS
  try:
    m.LEVELS = [art]
    return m.make_game(0)
  finally:
    m.LEVELS = saved


def ref_aperture_art(level):
  _import()
  from pycolab.examples import aperture as m
  return list(m.LEVELS[level])


def ref_storytelling():
  """The reference's storytelling module.  It spells `collections.Mapping` /
  `collections.Sequence` (gone since Python 3.10); alias them for the import —
  an environment shim, the reference source is untouched."""
  _import()
  import collections
  import collections.abc
  for name in ('Mapping', 'Sequence'):
    if not hasattr(collections, name):
      setattr(collections, name, getattr(collections.abc, name))
  from pycolab import storytelling
  return storytelling


def ref_warehouse(art, beneath=' ', level=None):
  m = _import()['warehouse_manager']
  if level is not None:
    return m.make_game(level)
  saved = (m.WAREHOUSES_ART, m.WAREHOUSES_WHAT_LIES_BENEATH)
  try:
    m.WAREHOUSES_ART = [art]
    m.WAREHOUSES_WHAT_LIES_BENEATH = [beneath]
    return m.make_game(0)
  finally:
    m.WAREHOUSES_ART, m.WAREHOUSES_WHAT_LIES_BENEATH = saved


def ref_stock_warehouse_art(level):
  m = _import()['warehouse_manager']
  wlb = m.WAREHOUSES_WHAT_LIES_BENEATH[level]
  return list(m.WAREHOUSES_ART[level]), (wlb if isinstance(wlb, str) else list(wlb))


def ref_marauders(art=None):
  m = _import()['extraterrestrial_marauders']
  if art is None:
    return m.make_game()
  saved = m.GAME_ART
  try:
    m.GAME_ART = art
    return m.make_game()
  finally:
    m.GAME_ART = saved


def ref_stock_marauders_art():
  return list(_import()['extraterrestrial_marauders'].GAME_ART)


_NAMES = ('n', 'ne', 'e', 'se', 's', 'sw', 'w', 'nw', 'stay')


def ref_fixture(art, what_lies_beneath, walkers, scrollys=None, drapes='',
                update_schedule=None, z_order=None, occlusion_in_layers=True):
  """Same signature as oracle.games.make_fixture_world, built from the
  reference's own test fixtures (tests/test_things.py)."""
  mods = _import()
  aa, tt = mods['ascii_art'], mods['test_things']
  scrollys = scrollys or {}
  sprites = {}
  for ch, kw in walkers.items():
    sprites[ch] = aa.Partial(
        tt.TestMazeWalker, impassable=kw.get('impassable', ''),
        confined_to_board=kw.get('confined', False),
        egocentric_scroller=kw.get('egocentric', False),
        scrolling_group=kw.get('group', ''))
  dr = {}
  shape = (len(art), len(art[0]))
  for ch, kw in scrollys.items():
    dr[ch] = aa.Partial(
        tt.TestScrolly, board_shape=shape,
        whole_pattern=np.array(kw['pattern'], dtype=bool),
        board_northwest_corner=tuple(kw['corner']),
        scroll_margins=kw.get('margins', (2, 3)),
        scrolling_group=kw.get('group', ''))
  for ch in drapes:
    dr[ch] = tt.TestDrape
  chars = list(walkers) + list(scrollys) + list(drapes)
  if update_schedule is None:
    update_schedule = [chars]
  return aa.ascii_art_to_game(art, what_lies_beneath, sprites, dr,
                              update_schedule=update_schedule, z_order=z_order,
                              occlusion_in_layers=occlusion_in_layers)


def fixture_actions_to_ref(actions):
  """Oracle motion codes -> the strings TestMazeWalker/TestScrolly expect."""
  if actions is None:
    return None
  if isinstance(actions, dict):
    return {ch: _NAMES[m] for ch, m in actions.items()}
  return _NAMES[actions]


def reward_pair(reward):
  """(value, has_reward) encoding used by fixtures and the device."""
  if reward is None:
    return 0, 0
  return int(reward), 1


def snapshot_things(engine):
  """{char: (row, col, visible)} for sprites of a reference engine."""
  out = {}
  for ch, ent in engine.things.items():
    if hasattr(ent, 'position'):
      out[ch] = (int(ent.position[0]), int(ent.position[1]), bool(ent.visible))
  return out


def _result_code(result):
  """A MazeWalker motion result in the oracle's encoding (engine_model.EDGE)."""
  from oracle import engine_model as em
  def code(x):
    return em.EDGE if x == 'edge!' else ord(x)
  if result is None:
    return None
  if isinstance(result, tuple):
    return tuple(code(x) for x in result)
  return code(result)


class ReferenceSide(object):
  """The original's engines for the scenarios of tests/reference_trace.py."""

  def scrolly_stock(self, level):
    return lambda: ref_scrolly_maze(None, None, level=level)

  def scrolly(self, maze, board, beneath):
    return lambda: ref_scrolly_maze(maze, board, beneath)

  def warehouse_stock(self, level):
    return lambda: ref_warehouse(None, level=level)

  def warehouse(self, art, beneath):
    return lambda: ref_warehouse(art, beneath)

  def marauders(self, seed):
    np.random.seed(seed)                  # the original draws from the global RNG
    return ref_marauders

  def fixture(self, art, walkers, scrollys=None, **kw):
    return ref_fixture(art, ' ', walkers, scrollys, **kw)

  def fixture_action(self, action):
    return fixture_actions_to_ref(action)

  def walk_result(self, engine, ch):
    return _result_code(engine.the_plot['walk_result_' + ch])

  def classic(self, kind, art):
    return lambda: ref_classic(kind, art)

  def aperture(self, level, art):
    return lambda: ref_aperture(level, art)

  def fluvial(self, art):
    art = art or ref_fluvial_art()
    return lambda: ref_fluvial(art)

  def scrolly_cropper(self, engine, pad, margins):
    crop = _import()['cropping'].ScrollingCropper(rows=9, cols=9, to_track=['P'],
                                                  scroll_margins=margins, pad_char=pad)
    crop.set_engine(engine)
    return lambda out: crop.crop(out[0]).board

  def ordeal(self):
    ref_storytelling()
    from pycolab.examples import ordeal
    return ordeal.make_game()

  def ordeal_chapter(self, story):
    return story.the_plot.this_chapter

  def apprehend(self, seed):
    import random
    _import()
    from pycolab.examples import apprehend
    random.seed(seed)
    return apprehend.make_game()

  def ball_registers(self, engine):
    ball = engine.things['b']
    return float(ball._dx), float(ball._x_accumulator)

  def shockwave(self, art, seed):
    _import()
    from pycolab.examples import shockwave as m
    np.random.seed(seed)
    saved = m.LEVELS
    try:
      m.LEVELS = [art]
      return m.make_game(0)
    finally:
      m.LEVELS = saved

  def shockwave_stock_art(self):
    _import()
    from pycolab.examples import shockwave as m
    return m.LEVELS[0]
