"""Differential tests: oracle restatement vs the original pycolab.

These pin the oracle (`oracle/`) to the original on seeded random action streams
for every configured game, on stock and generated levels, plus random walks of
the original's own MazeWalker/Scrolly test fixtures.  The original's side of
each comparison is stored in tests/golden/reference_traces.npz (see
tests/reference_trace.py and tests/golden/make_reference_traces.py).
"""

import os

import numpy as np
import pytest

import reference_trace as rt
from oracle import games

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                      'reference_traces.npz')


def _check(key, scenario, *args):
  """Replay one scenario on the oracle; its trace must be the original's."""
  with np.load(GOLDEN) as z:
    want = z[key]
  trace, facts = scenario(rt.ORACLE, *args)
  got = trace.result()
  assert got[-1] == want[-1], '%s: %d records, the original made %d' % (key, got[-1], want[-1])
  bad = np.flatnonzero(got != want)
  assert not len(bad), '%s: first difference within records %d..%d' % (
      key, bad[0] * rt.Trace.EVERY, min((bad[0] + 1) * rt.Trace.EVERY, int(want[-1])))
  return facts


def test_every_scenario_has_a_stored_trace():
  with np.load(GOLDEN) as z:
    assert sorted(z.files) == sorted(rt.cases())


@pytest.mark.parametrize('level', [0, 1, 2])
def test_scrolly_maze_stock(level):
  _check('scrolly_stock_%d' % level, rt.scrolly_stock, level)


def test_scrolly_maze_stock_with_quit():
  assert _check('scrolly_stock_with_quit', rt.scrolly_stock_with_quit)['episodes'] > 10


@pytest.mark.parametrize('seed', [0, 1])
def test_scrolly_maze_generated_64(seed):
  _check('scrolly_generated_64_%d' % seed, rt.scrolly_generated_64, seed)


@pytest.mark.parametrize('level', [0, 1, 2])
def test_warehouse_stock(level):
  _check('warehouse_stock_%d' % level, rt.warehouse_stock, level)


def test_warehouse_generated_80():
  _check('warehouse_generated_80', rt.warehouse_generated_80)


def test_marauders_layout_matches_stock():
  from pycolab_b200 import levels
  art = levels.marauders_level()
  with np.load(os.path.join(os.path.dirname(GOLDEN), 'marauders_stock_s0.npz')) as z:
    assert art == [bytes(r).decode('ascii') for r in z['art']]


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_marauders_stock(seed):
  # The original draws from the GLOBAL NumPy RNG seeded once, the oracle from its
  # own RandomState(seed); episodes continue the same stream.
  assert _check('marauders_stock_%d' % seed, rt.marauders_stock, seed)['episodes'] >= 1


@pytest.mark.parametrize('seed', range(8))
def test_fixture_walkers_random(seed):
  _check('fixture_walkers_%d' % seed, rt.fixture_walkers_random, seed)


@pytest.mark.parametrize('seed,margins', rt.FIXTURE_SCROLLY)
def test_fixture_scrolly_random(seed, margins):
  raised_at = _check('fixture_scrolly_%d' % seed, rt.fixture_scrolly_random, seed,
                     margins)['raised_at']
  assert raised_at is None or raised_at > 3


@pytest.mark.parametrize('kind', games.CLASSIC_KINDS)
@pytest.mark.parametrize('art', ['stock', 'other'])
def test_classics(kind, art):
  facts = _check('classic_%s_%s' % (kind, art), rt.classics, kind, art)
  assert facts['episodes'] >= 1 and facts['rewards'] > 0


@pytest.mark.parametrize('level', [0, 1, 2, 'other'])
def test_aperture_stock(level):
  assert _check('aperture_%s' % level, rt.aperture, level)['shots'] > 100


@pytest.mark.parametrize('art', ['stock', 'other'])
def test_fluvial_natation(art):
  assert _check('fluvial_%s' % art, rt.fluvial_natation, art)['episodes'] > 5


@pytest.mark.parametrize('pad,margins', rt.CROPPERS)
def test_scrolling_cropper(pad, margins):
  _check('cropper_%d' % rt.CROPPERS.index((pad, margins)), rt.scrolling_cropper, pad, margins)


@pytest.mark.parametrize('seed', range(6))
def test_ordeal_story_random_walks(seed):
  """examples/ordeal.py: the original's Story vs the chained oracle worlds,
  random walks across all three sub-games."""
  _check('ordeal_%d' % seed, rt.ordeal_story, seed)


def test_apprehend_many_episodes():
  """examples/apprehend.py: 200 episodes, the oracle drawing from
  random.Random(seed) what the original draws from the seeded global `random`."""
  facts = _check('apprehend', rt.apprehend_many_episodes)
  assert facts['steps'] > 1500 and facts['wins'] > 20


@pytest.mark.parametrize('level', ['stock', 'generated'])
def test_shockwave_many_episodes(level):
  facts = _check('shockwave_%s' % level, rt.shockwave_many_episodes, level)
  assert facts['steps'] > 400 and facts['ends'] > 60
