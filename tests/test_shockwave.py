"""examples/shockwave.py (SURVEY.md §8f-4): a walker, two static drapes and a ring of
fire around `np.random.randint` impact points whose update() reads the STALE board.
Goldens are the reference's own trajectories (tests/golden/shockwave_*: the stock level
and two generated ones, policy-driven so that some episodes are won); CPU: the oracle;
GPU: the facade Engine (B = 1, global NumPy generator handed to the device) and a
batched lock-step with per-env generators."""

import os

import numpy as np
import pytest

import golden_cases as gc
import reference_trace as rt
import trajectory as tj
from oracle import games as ogames

NAMES = gc.names('shockwave_')


def _rows(env):
  s = env.things['P']
  vp = getattr(s, 'virtual_position', s.position)
  return [[int(s.position[0]), int(s.position[1]), int(bool(s.visible)), int(vp[0]), int(vp[1])]]


@pytest.mark.parametrize('name', NAMES)
def test_oracle_shockwave_matches_reference_golden(name):
  g = gc.load(name)
  art = tj.u8_to_art(g['art'])
  rng = np.random.RandomState(int(g['numpy_seed'][0]))
  sprites, curtains = [], []

  def on_frame(env, out):
    sprites.append(_rows(env))
    curtains.append(env.things['@'].curtain.copy())
  got = tj.run_trajectory(lambda: ogames.make_shockwave(art, rng), g['actions'].tolist(),
                          on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  np.testing.assert_array_equal(g['sprites'], np.array(sprites))
  np.testing.assert_array_equal(g['curtains'].astype(bool), np.stack(curtains))
  assert int((g['reward'] == 1).sum()) >= 1          # the safe-zone path is on the tape


@pytest.mark.gpu
@pytest.mark.parametrize('name', NAMES)
def test_facade_shockwave_golden(name):
  from pycolab_b200.games import shockwave
  g = gc.load(name)
  art = tj.u8_to_art(g['art'])
  sprites, curtains = [], []

  def on_frame(env, out):
    sprites.append(_rows(env))
    curtains.append(np.asarray(env.things['@'].curtain).copy())
  np.random.seed(int(g['numpy_seed'][0]))
  got = tj.run_trajectory(lambda: shockwave.make_game(art), g['actions'].tolist(),
                          on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  np.testing.assert_array_equal(g['sprites'], np.array(sprites))
  np.testing.assert_array_equal(g['curtains'].astype(bool), np.stack(curtains))


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(12, 15), (32, 64), (9, 33)])
def test_batched_shockwave_vs_oracle(shape):
  """Auto-resetting batch over several generated levels, one NumPy generator per env
  (RandomState(seed + e)), boards / curtains / rewards / discounts every step."""
  import torch
  from pycolab_b200 import batched, levels
  from pycolab_b200.games import shockwave
  arts = [levels.shockwave_level(30 + i, shape[0], shape[1], 0.45) for i in range(3)]
  B, T, seed = 13, 220, 9
  eng = batched.BatchedEngine([shockwave.make_game(a) for a in arts], batch=B, rng_seed=seed)
  rngs = [np.random.RandomState(seed + e) for e in range(B)]
  make = lambda e: ogames.make_shockwave(arts[e % len(arts)], rngs[e])
  worlds = [make(e) for e in range(B)]
  outs = [w.its_showtime() for w in worlds]
  res = eng.its_showtime()
  rs = np.random.RandomState(4)
  episodes = wins = 0
  for t in range(T + 1):
    torch.cuda.synchronize()
    boards = res.board.cpu().numpy()
    cur = eng.curtain('@').cpu().numpy()
    for e in range(B):
      np.testing.assert_array_equal(boards[e][:, :shape[1]], outs[e][0],
                                    err_msg='t=%d env=%d' % (t, e))
      np.testing.assert_array_equal(cur[e], worlds[e].things['@'].curtain)
      want = outs[e][1]
      assert (int(res.has_reward[e]), int(res.reward[e])) == (
          (0, 0) if want is None else (1, int(want))), (t, e)
      assert float(res.discount[e]) == float(outs[e][2])
      assert bool(res.done[e]) == worlds[e].game_over
    if t == T:
      break
    act = rs.choice([0, 1, 2, 3, 4], size=B, p=[.6, .12, .12, .12, .04]).astype(np.int32)
    res = eng.play(torch.from_numpy(act).cuda())
    for e in range(B):
      if worlds[e].game_over:
        episodes += 1
        wins += outs[e][1] == 1
        worlds[e] = make(e)
        outs[e] = worlds[e].its_showtime()
      else:
        outs[e] = worlds[e].play(int(act[e]))
  assert episodes > B
  assert int(eng.error_codes().abs().max()) == 0


def test_shockwave_lowers_and_validates_on_cpu():
  import ctypes as C
  from pycolab_b200 import _lib, errors, levels, lowering
  from pycolab_b200.games import shockwave
  game = lowering.lower(shockwave.make_game(0))
  assert game.program == _lib.PROG_SHOCKWAVE and game.drape_chars == '@ ^'
  assert game.needs_rng and game.rng_kind == 'numpy' and game.program_arg[0] == 2
  lib = _lib.load()
  handle = C.c_void_p()
  spec = game.make_spec(True)
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(handle)) == _lib.OK
  lib.pcl_destroy(handle)
  spec.rows = 40                                   # one curtain row per lane: 32 rows at most
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(handle)) != _lib.OK
  with pytest.raises(errors.NotLoweredError):
    lowering.lower(shockwave.make_game(levels.shockwave_level(0, 40, 20)))


def test_reference_shockwave_file_lowers_like_the_twin():
  """The original's examples/shockwave.py, loaded through `compat`, lowered to
  what this package's twin lowers to."""
  from pycolab_b200 import lowering
  from pycolab_b200.games import shockwave
  rt.check_lowering('shockwave', lowering.lower(shockwave.make_game(0)))
