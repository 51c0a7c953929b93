"""examples/ordeal.py (SURVEY.md §8f-4): a `storytelling.Story` of three sub-games
whose entities carry `has_sword` / `last_position` across chapters in the Plot and
issue `Plot.change_z_order` on a real game (ordeal.py:182-185).

Goldens (tests/golden/ordeal_*.npz) are the reference's own Story on BFS-scripted
walks (sword + victory, no sword + defeat, castle and back, quit) and random walks.
CPU: the oracle restatement chained like Story does; GPU: this package's Story over
device-backed Engines and the device cropper; plus, where an upstream pycolab
checkout is named by PYCOLAB_UPSTREAM, its unmodified ordeal.py loaded through
`compat`.
"""

import os

import numpy as np
import pytest

import golden_cases as gc
import reference_trace as rt
import refdriver
import trajectory as tj
from oracle import engine_model as em
from oracle import games as ogames

NAMES = gc.names('ordeal_')


class OracleOrdeal(object):
  """The three oracle worlds chained the way Story chains Engines
  (storytelling.py:391-474): crop, start successors until one survives its first
  frame, sum the rewards, keep the last discount."""

  def __init__(self):
    from pycolab_b200.games import ordeal
    self._arts = ordeal.ARTS
    self._crop = em.ScrollingCrop(8, 15, ['P'], scroll_margins=(2, 3))
    self.game_over = False
    self._enter('kansas', None)

  def _enter(self, chapter, story_plot):
    self.world = ogames.make_ordeal(chapter, self._arts[chapter], story_plot)
    self.chapter = chapter
    if chapter == 'kansas':
      self._crop.set_engine(self.world)

  def _view(self, board):
    return self._crop.crop(board) if self.chapter == 'kansas' else board

  def _deliver(self, out):
    board, reward, discount = out
    view = self._view(board)
    while self.world.game_over:
      store = self.world.plot.store
      if store['next_chapter'] is None:
        self.game_over = True
        break
      self._enter(store['next_chapter'], dict(has_sword=store['has_sword'],
                                              last_position=store['last_position'],
                                              prior_chapter=store['this_chapter']))
      board, more, discount = self.world.its_showtime()
      view = self._view(board)
      if more is not None:
        reward = more if reward is None else reward + more
    return view, reward, discount

  def its_showtime(self):
    return self._deliver(self.world.its_showtime())

  def play(self, action):
    return self._deliver(self.world.play(action))


@pytest.mark.parametrize('name', NAMES)
def test_oracle_ordeal_matches_reference_golden(name):
  g = gc.load(name)
  chapters, swords = [], []

  def on_frame(env, out):
    chapters.append(env.chapter)
    swords.append(1 if env.world.plot.store.get('has_sword') else 0)
  got = tj.run_trajectory(OracleOrdeal, g['actions'].tolist(), on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  assert chapters == g['chapters'].tolist()
  assert swords == g['has_sword'].tolist()


def test_goldens_cover_the_interesting_paths():
  wins, loses = gc.load('ordeal_sword_wins'), gc.load('ordeal_no_sword_loses')
  assert wins['reward'].sum() == 2 and set(wins['chapters'].tolist()) == {'kansas', 'cavern',
                                                                          'castle'}
  assert loses['reward'].sum() == -1 and loses['has_sword'].max() == 0
  assert wins['has_sword'].max() == 1 and int(wins['game_over'].sum()) >= 1


def _run_device_story(name, make_story):
  g = gc.load(name)
  chapters, swords = [], []

  def on_frame(env, out):
    chapters.append(str(env.the_plot.this_chapter))
    swords.append(1 if env.the_plot.get('has_sword') else 0)
  got = tj.run_trajectory(make_story, g['actions'].tolist(), on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  assert chapters == g['chapters'].tolist()
  assert swords == g['has_sword'].tolist()


@pytest.mark.gpu
@pytest.mark.parametrize('name', NAMES)
def test_device_ordeal_story_matches_reference_golden(name):
  from pycolab_b200.games import ordeal
  _run_device_story(name, ordeal.make_game)


@pytest.mark.gpu
def test_device_ordeal_z_order_follows_the_battle():
  """ordeal.py:182-185 on the device: the winner is drawn on top."""
  from pycolab_b200.games import ordeal
  for name, front in (('ordeal_sword_wins', 'D'), ('ordeal_no_sword_loses', 'P')):
    g = gc.load(name)
    story = ordeal.make_game()
    story.its_showtime()
    for a in g['actions'].tolist():
      story.play(a)
      if story.game_over:
        break
    assert story.game_over and story.the_plot.this_chapter == 'castle'
    assert story.current_game.z_order[-1] == front, name


@pytest.mark.gpu
@pytest.mark.skipif(not refdriver.available(), reason=refdriver.MISSING)
def test_reference_ordeal_file_runs_on_the_device_through_compat():
  """The reference's own examples/ordeal.py, unmodified: its classes subclass this
  package's prefabs, `lowering` recognises them by source fingerprint, and its
  `make_game()` Story runs on device-backed Engines."""
  import sys
  from pycolab_b200 import compat
  saved = {k: v for k, v in sys.modules.items() if k == 'pycolab' or k.startswith('pycolab.')}
  compat.uninstall()
  try:
    mod = compat.load_example(os.path.join(refdriver.REFERENCE_ROOT, 'pycolab', 'examples',
                                           'ordeal.py'))
    _run_device_story('ordeal_sword_wins', mod.make_game)
  finally:
    compat.uninstall()
    sys.modules.update(saved)


def test_reference_ordeal_chapters_lower_like_the_twins():
  """The chapters the original's examples/ordeal.py builds (with its classes and
  art, ordeal.py:77-93), loaded through `compat`, lowered to what this package's
  chapters lower to."""
  from pycolab_b200 import lowering
  from pycolab_b200.games import ordeal
  mine = {'castle': ordeal.make_castle(), 'cavern': ordeal.make_cavern(),
          'kansas': ordeal.make_kansas()}
  for chapter, game in mine.items():
    rt.check_lowering('ordeal_' + chapter, lowering.lower(game))
