"""Observation post-processors: oracle vs the original (CPU), device vs oracle (GPU)."""

import os

import numpy as np
import pytest

import golden_cases as gc
from oracle import engine_model as em

WAREHOUSE_REPAINT = {c: 'x' for c in '0123456789'}
RGB = {' ': (0, 0, 0), '.': (9, 9, 9), '#': (200, 0, 250), '_': (1, 2, 3), 'P': (0, 255, 255),
       'X': (250, 100, 50)}
RGB.update({c: (180, 100, 10) for c in '0123456789'})


def _boards(name, n=6):
  g = gc.load(name)
  idx = np.linspace(0, len(g['boards']) - 1, n).astype(int)
  return g['boards'][idx]


def observer_outputs(module, boards):
  """{name: array} of the post-processors of `module` (the original's
  `pycolab.rendering` or `oracle_rendering` below) on `boards`."""
  out = {}
  chars = set(' .#_PX0123456789')
  scalar = {c: float(ord(c)) / 2 for c in chars}
  for i, board in enumerate(boards):
    obs = module.Observation(board=board, layers={c: board == ord(c) for c in chars})
    out['repaint_%d' % i] = module.ObservationCharacterRepainter(WAREHOUSE_REPAINT)(obs).board
    for permute in (None, (1, 2, 0), (2, 0, 1)):
      tag = '%d_%s' % (i, ''.join(map(str, permute or ())))
      out['rgb_' + tag] = module.ObservationToArray(RGB, dtype=np.uint8, permute=permute)(obs)
      out['features_' + tag] = module.ObservationToFeatureArray('P#_0X', permute=permute)(obs)
    out['scalar_%d' % i] = module.ObservationToArray(scalar, dtype=np.float32,
                                                     permute=(1, 0))(obs)
  return out


class oracle_rendering(object):
  """The oracle's post-processors behind the original's class names."""
  class Observation(object):
    def __init__(self, board, layers):
      self.board = board

  class ObservationCharacterRepainter(object):
    def __init__(self, mapping):
      self.mapping = mapping

    def __call__(self, obs):
      return oracle_rendering.Observation(em.observation_repaint(obs.board, self.mapping), None)

  class ObservationToArray(object):
    def __init__(self, value_mapping, dtype, permute):
      self.args = value_mapping, dtype, permute

    def __call__(self, obs):
      return em.observation_to_array(obs.board, *self.args)

  class ObservationToFeatureArray(object):
    def __init__(self, layers, permute):
      self.args = layers, permute

    def __call__(self, obs):
      return em.observation_to_feature_array(obs.board, *self.args)


def test_oracle_post_processors_match_reference():
  """Against the original's outputs, stored in tests/golden/reference_observers.npz
  by tests/golden/make_reference_traces.py."""
  with np.load(os.path.join(gc.GOLDEN_DIR, 'reference_observers.npz')) as z:
    want = {k: z[k] for k in z.files}
  got = observer_outputs(oracle_rendering, _boards('warehouse_stock_L1'))
  assert sorted(got) == sorted(want)
  for k in want:
    np.testing.assert_array_equal(got[k], want[k], err_msg=k)


@pytest.mark.gpu
def test_facade_post_processors_vs_oracle():
  from pycolab_b200 import rendering
  for board in _boards('warehouse_stock_L1'):
    chars = set(' .#_PX0123456789')
    obs = rendering.Observation(board=board, layers=rendering.LazyLayers(board, chars))
    rep = rendering.ObservationCharacterRepainter(WAREHOUSE_REPAINT)(obs)
    np.testing.assert_array_equal(rep.board, em.observation_repaint(board, WAREHOUSE_REPAINT))
    assert set(rep.layers) == (chars - set('0123456789')) | {'x'}
    np.testing.assert_array_equal(rep.layers['x'], rep.board == ord('x'))
    for permute in (None, (1, 2, 0), (2, 0, 1), (0, 2, 1)):
      got = rendering.ObservationToArray(RGB, dtype=np.uint8, permute=permute)(obs)
      want = em.observation_to_array(board, RGB, np.uint8, permute)
      assert got.dtype == want.dtype and got.shape == want.shape
      np.testing.assert_array_equal(got, want)
      got = rendering.ObservationToFeatureArray('P#_0X', permute=permute)(obs)
      want = em.observation_to_feature_array(board, 'P#_0X', permute)
      assert got.dtype == np.float32 and got.shape == want.shape
      np.testing.assert_array_equal(got, want)
    scalar = {c: float(ord(c)) / 2 for c in chars}
    np.testing.assert_array_equal(
        rendering.ObservationToArray(scalar, dtype=np.float32, permute=(1, 0))(obs),
        em.observation_to_array(board, scalar, np.float32, (1, 0)))
  # error behaviour (rendering.py:449-470, 520-526, 590-596)
  with pytest.raises(ValueError):
    rendering.ObservationToArray(RGB, permute=(0, 1))
  with pytest.raises(ValueError):
    rendering.ObservationToFeatureArray('P', permute=(0, 1))
  with pytest.raises(RuntimeError):
    rendering.ObservationToArray({' ': 0, '#': 1})(obs)
  with pytest.raises(RuntimeError):
    rendering.ObservationToFeatureArray('QZ')(obs)


@pytest.mark.gpu
def test_batched_post_processors_vs_oracle():
  import torch
  from pycolab_b200 import batched, levels
  from pycolab_b200.games import scrolly_maze
  arts = [levels.scrolly_maze_level(50 + i, world_shape=(65, 65), board_shape=(30, 45))
          for i in range(3)]
  eng = batched.BatchedEngine([scrolly_maze.make_game(*a) for a in arts], batch=9)
  eng.its_showtime()
  rs = np.random.RandomState(0)
  for _ in range(12):
    eng.play(torch.from_numpy(rs.randint(0, 5, size=9).astype(np.int32)).cuda())
  boards = eng.board.cpu().numpy()
  feats = eng.to_feature_array('P#@ab', permute=(1, 2, 0)).cpu().numpy()
  assert feats.shape == (9, 30, 45, 5) and feats.dtype == np.float32
  rgb = {c: (i, 2 * i, 255 - i) for i, c in enumerate(' .#@Pabc')}
  arr = eng.to_array(rgb, dtype=np.uint8).cpu().numpy()
  rep = eng.repaint({'a': 'e', 'b': 'e', 'c': 'e'}).cpu().numpy()
  for e in range(9):
    np.testing.assert_array_equal(feats[e],
                                  em.observation_to_feature_array(boards[e], 'P#@ab', (1, 2, 0)))
    np.testing.assert_array_equal(arr[e], em.observation_to_array(boards[e], rgb, np.uint8))
    np.testing.assert_array_equal(rep[e], em.observation_repaint(
        boards[e], {'a': 'e', 'b': 'e', 'c': 'e'}))
  with pytest.raises(RuntimeError):
    eng.to_array({' ': 0.0, '#': 1.0})
