"""`storytelling.Story` (host-side caller of the path) on CPU.

The Story logic is driven here by oracle Worlds dressed as Engines, against the
golden trajectory the reference's own Story produced for the same chapters
(tests/golden/story_classics_list.npz); plus the constructor's argument checks
(storytelling.py:493-622).
"""

import importlib

import numpy as np
import pytest

import golden_cases as gc
import story_cases
import trajectory as tj
from oracle import games as ogames
from pycolab_b200 import engine as engine_lib
from pycolab_b200 import plot as plot_lib
from pycolab_b200 import rendering
from pycolab_b200 import storytelling
from pycolab_b200 import things


class _Walker(things.Sprite):
  def update(self, *args, **kwargs):
    raise AssertionError('never called')


class OracleEngine(object):
  """An oracle World with the attributes Story reads from an Engine."""

  def __init__(self, world, palette):
    self._world = world
    self.the_plot = plot_lib.Plot()
    self.rows, self.cols = world.rows, world.cols
    self._palette = palette

  def _obs(self, out):
    board = np.asarray(out[0], dtype=np.uint8)
    chars = set(self._palette) | set(self._world.things)
    return rendering.Observation(board=board, layers=rendering.LazyLayers(board, chars)), out[1], out[2]

  def its_showtime(self):
    return self._obs(self._world.its_showtime())

  def play(self, actions):
    return self._obs(self._world.play(actions))

  @property
  def game_over(self):
    return self._world.game_over

  @property
  def z_order(self):
    return list(self._world.things)

  @property
  def backdrop(self):
    return things.Backdrop(curtain=self._world.backdrop, palette=engine_lib.Palette(self._palette))

  @property
  def things(self):
    return {ch: _Walker(things.Sprite.Position(self.rows, self.cols),
                        things.Sprite.Position(w.row, w.col), ch)
            for ch, w in self._world.things.items()}


def _oracle_chapter(kind, art):
  stock = importlib.import_module('pycolab_b200.games.classics.' + kind).GAME_ART
  palette = ' #' if kind == 'four_rooms' else '.'
  return lambda: OracleEngine(ogames.make_classic(kind, art or list(stock)), palette)


def test_list_story_matches_reference_golden():
  g = gc.load('story_classics_list')
  chapters = []
  make = lambda: storytelling.Story([_oracle_chapter(k, a) for k, a in story_cases.LIST_CHAPTERS])
  got = tj.run_trajectory(make, g['actions'].tolist(),
                          on_frame=lambda env, out: chapters.append(str(env.the_plot.this_chapter)))
  tj.assert_same_trajectory(g, got, 'story_classics_list')
  assert chapters == g['chapters'].tolist()


def test_story_views_and_plot_hand_over():
  story = storytelling.Story([_oracle_chapter(k, a) for k, a in story_cases.LIST_CHAPTERS])
  story.its_showtime()
  assert (story.rows, story.cols) == (4, 12)
  assert story.z_order == ['P'] and set(story.backdrop.palette) == {'.'}
  assert not storytelling.is_fictional(story.things['P'])
  story.the_plot['note'] = 42
  first = story.current_game
  # one step east falls off the cliff: chapter 0 ends, chapter 1 starts in the same call
  obs, reward, discount = story.play(3)
  assert first.game_over and story.current_game is not first and not story.game_over
  assert story.the_plot['note'] == 42                       # Plot entries travel
  assert (story.the_plot.prior_chapter, story.the_plot.this_chapter,
          story.the_plot.next_chapter) == (0, 1, 2)
  assert reward == -100.0 and discount == 1.0               # new game's discount, old reward
  with pytest.raises(RuntimeError):
    story.its_showtime()


def test_story_ends_after_last_chapter_and_refuses_more_play():
  story = storytelling.Story([_oracle_chapter('chain_walk', None)])
  story.its_showtime()
  for _ in range(2):
    obs, reward, discount = story.play(0)
  assert story.game_over and reward == 1.0 and discount == 0.0
  with pytest.raises(RuntimeError):
    story.play(0)


def test_dict_story_follows_next_chapter_and_rejects_unknown_keys():
  def cliff_then(target):
    def build():
      game = _oracle_chapter('cliff_walk', None)()
      game.the_plot.next_chapter = target
      return game
    return build
  story = storytelling.Story({'a': cliff_then('b'), 'b': cliff_then(None)}, first_chapter='a')
  story.its_showtime()
  story.play(3)
  assert story.the_plot.this_chapter == 'b' and story.the_plot.prior_chapter == 'a'
  bad = storytelling.Story({'a': cliff_then('nowhere')}, first_chapter='a')
  bad.its_showtime()
  with pytest.raises(KeyError):
    bad.play(3)


def test_constructor_argument_checks():
  rooms, cliff = _oracle_chapter('four_rooms', None), _oracle_chapter('cliff_walk', None)
  with pytest.raises(ValueError):
    storytelling.Story([])
  with pytest.raises(ValueError):
    storytelling.Story({None: cliff}, first_chapter=None)
  with pytest.raises(ValueError):
    storytelling.Story({'a': cliff}, first_chapter='b')
  with pytest.raises(ValueError):
    storytelling.Story([cliff, cliff], croppers=[None])          # keys differ
  with pytest.raises(ValueError):
    storytelling.Story([rooms, cliff])                           # 13x13 vs 4x12 observations

  class _DrapeP(OracleEngine):                                   # 'P' as a Drape elsewhere
    @property
    def things(self):
      class D(things.Drape):
        def update(self, *args, **kwargs):
          pass
      return {'P': D(np.zeros((self.rows, self.cols), dtype=bool), 'P')}
  clash = lambda: _DrapeP(ogames.make_classic('cliff_walk', ['............'] * 3 + ['P...........']), '.')
  with pytest.raises(ValueError):
    storytelling.Story([cliff, clash])


def test_reference_story_tests_pass_against_this_story_class():
  """The behaviours the original's tests/story_test.py checks, on this package's
  Story over oracle and scripted chapters: a sequence and a dict of games,
  cropping, rewards carried across chapter changes (and the summing test below),
  stand-ins and the merged backdrop palette for characters of other chapters,
  and refusal of a character used in two different ways."""
  from pycolab_b200 import cropping

  class CornerCropper(cropping.ObservationCropper):    # a host-side FixedCropper((0, 0), ...)
    def __init__(self, rows, cols):
      super(CornerCropper, self).__init__()
      self._shape = rows, cols

    def crop(self, observation):
      board = np.ascontiguousarray(observation.board[:self._shape[0], :self._shape[1]])
      return rendering.Observation(board=board, layers=rendering.LazyLayers(board, '.# P'))

    @property
    def rows(self):
      return self._shape[0]

    @property
    def cols(self):
      return self._shape[1]

  # a sequence of games is played in order, to the end of the last one
  g = gc.load('story_classics_list')
  story = storytelling.Story([_oracle_chapter(k, a) for k, a in story_cases.LIST_CHAPTERS])
  story.its_showtime()
  seen = [story.the_plot.this_chapter]
  for a in g['actions'].tolist():
    if story.game_over:
      break
    story.play(a)
    seen.append(story.the_plot.this_chapter)
  assert sorted(set(seen)) == [0, 1, 2] and seen == sorted(seen) and story.game_over

  # a dict of games follows Plot.next_chapter; the finished game's reward is
  # delivered with the successor's first frame
  def cliff_then(target):
    def build():
      game = _oracle_chapter('cliff_walk', None)()
      game.the_plot.next_chapter = target
      return game
    return build
  story = storytelling.Story({'x': cliff_then('y'), 'y': cliff_then(None)}, first_chapter='x')
  story.its_showtime()
  obs, reward, _ = story.play(3)                               # off the cliff
  assert story.the_plot.this_chapter == 'y' and reward == -100.0 and not story.game_over

  # croppers apply per chapter, and chapters of another shape are then compatible
  rooms, cliff = _oracle_chapter('four_rooms', None), _oracle_chapter('cliff_walk', None)
  with pytest.raises(ValueError):
    storytelling.Story([rooms, cliff])
  story = storytelling.Story([rooms, cliff], croppers=[CornerCropper(3, 4), CornerCropper(3, 4)])
  obs, _, _ = story.its_showtime()
  assert obs.board.shape == (3, 4) and (story.rows, story.cols) == (3, 4)
  np.testing.assert_array_equal(obs.board, rooms().its_showtime()[0].board[:3, :4])

  # characters of other chapters get invisible stand-ins below the current z-order,
  # and the backdrop palette is every chapter's backdrop characters
  story = storytelling.Story([_ScriptedChapter(sprites='a', drapes='X', palette=' #'),
                              _ScriptedChapter(sprites='b', palette=' .', first_reward=None)])
  story.its_showtime()
  assert set(story.backdrop.palette) == {' ', '#', '.'}
  assert set(story.things) == {'a', 'b', 'X'}
  assert not storytelling.is_fictional(story.things['a'])
  assert not storytelling.is_fictional(story.things['X'])
  assert storytelling.is_fictional(story.things['b']) and not story.things['b'].visible
  assert story.z_order == ['b', 'X', 'a']
  story.play(0)                                                 # chapter 0 ends
  assert story.the_plot.this_chapter == 1
  assert set(story.things) == {'a', 'b', 'X'}
  assert not storytelling.is_fictional(story.things['b'])
  assert storytelling.is_fictional(story.things['a']) and not story.things['a'].visible
  assert storytelling.is_fictional(story.things['X']) and not story.things['X'].curtain.any()

  # a character used in two different ways across chapters is refused
  for one, other in [(dict(sprites='a'), dict(drapes='a')),
                     (dict(sprites='#'), dict(palette=' #')),
                     (dict(drapes='#'), dict(palette=' #'))]:
    with pytest.raises(ValueError, match='same character in two different ways'):
      storytelling.Story([_ScriptedChapter(**one), _ScriptedChapter(**other)])


def test_rewards_of_chapters_that_end_on_their_first_frame_are_summed():
  """A finished chapter's successors are started one after another until one
  survives its first frame; the finished chapter's reward and every successor's
  first-frame reward arrive summed in the same step, with the last started
  chapter's discount."""
  chapters = [_ScriptedChapter(first_reward=None, rewards=[2.0]),
              _ScriptedChapter(first_reward=4.0, rewards=[]),       # over on its first frame
              _ScriptedChapter(first_reward=8.0, rewards=[]),       # ... and so is this one
              _ScriptedChapter(first_reward=1.0, rewards=[5.0], discount=0.5)]
  story = storytelling.Story(chapters)
  obs, reward, discount = story.its_showtime()
  assert reward is None and story.the_plot.this_chapter == 0
  obs, reward, discount = story.play(0)
  assert reward == 15.0 and discount == 0.5
  assert story.the_plot.this_chapter == 3 and not story.game_over
  obs, reward, discount = story.play(0)
  assert reward == 5.0 and discount == 0.0 and story.game_over


class _ScriptedChapter(object):
  """Builder of a tiny Engine-like chapter with a scripted outcome: its_showtime()
  yields `first_reward` (and ends the game at once when `rewards` is empty), then
  each play() yields the next of `rewards`; the last one ends the game with
  discount 0.  Entities: sprites at the top-left, drapes with empty curtains."""

  def __init__(self, sprites='', drapes='', palette=' ', first_reward=None, rewards=(1.0,),
               discount=1.0):
    self.kw = dict(sprites=sprites, drapes=drapes, palette=palette, first_reward=first_reward,
                   rewards=list(rewards), discount=discount)

  def __call__(self):
    return _ScriptedEngine(**self.kw)


class _ScriptedEngine(object):
  rows, cols = 2, 3

  def __init__(self, sprites, drapes, palette, first_reward, rewards, discount):
    self.the_plot = plot_lib.Plot()
    self._palette, self._first, self._rewards, self._discount = (
        palette, first_reward, rewards, discount)
    corner = things.Sprite.Position(self.rows, self.cols)
    self._things = {ch: _Walker(corner, things.Sprite.Position(0, 0), ch) for ch in sprites}
    for ch in drapes:
      self._things[ch] = _Curtain(np.zeros((self.rows, self.cols), dtype=bool), ch)
    self.game_over = False

  def _out(self, reward, discount):
    board = np.full((self.rows, self.cols), ord(self._palette[0]), dtype=np.uint8)
    obs = rendering.Observation(board=board, layers=rendering.LazyLayers(board, self._palette))
    return obs, reward, discount

  def its_showtime(self):
    self.game_over = not self._rewards
    return self._out(self._first, 0.0 if self.game_over else self._discount)

  def play(self, actions):
    reward = self._rewards.pop(0)
    self.game_over = not self._rewards
    return self._out(reward, 0.0 if self.game_over else self._discount)

  @property
  def z_order(self):
    return sorted(self._things)

  @property
  def backdrop(self):
    board = np.full((self.rows, self.cols), ord(self._palette[0]), dtype=np.uint8)
    return things.Backdrop(curtain=board, palette=engine_lib.Palette(self._palette))

  @property
  def things(self):
    return dict(self._things)


class _Curtain(things.Drape):
  def update(self, *args, **kwargs):
    raise AssertionError('never called')
