"""examples/apprehend.py (SURVEY.md §8f-4): two MazeWalkers, a float64 accumulator and
one draw from Python's `random` per episode.  Goldens are the reference's own
trajectories (tests/golden/apprehend_stock_*: 30 episodes each, `random.seed` fixed);
CPU: the oracle; GPU: the facade Engine (B = 1, slopes drawn by the Python sprites) and
a batched lock-step whose slopes are drawn ON THE DEVICE from per-env MT19937 states."""

import os
import random

import numpy as np
import pytest

import golden_cases as gc
import reference_trace as rt
import trajectory as tj
from oracle import games as ogames

NAMES = gc.names('apprehend_')


def _rows(env, chars='Pb'):
  out = []
  for ch in chars:
    s = env.things[ch]
    vp = getattr(s, 'virtual_position', s.position)
    out.append([int(s.position[0]), int(s.position[1]), int(bool(s.visible)),
                int(vp[0]), int(vp[1])])
  return out


@pytest.mark.parametrize('name', NAMES)
def test_oracle_apprehend_matches_reference_golden(name):
  g = gc.load(name)
  art = tj.u8_to_art(g['art'])
  rng = random.Random(int(g['random_seed'][0]))
  sprites, floats = [], []

  def on_frame(env, out):
    sprites.append(_rows(env))
    floats.append([env.things['b'].aux['dx'], env.things['b'].aux['acc']])
  got = tj.run_trajectory(lambda: ogames.make_apprehend(art, rng), g['actions'].tolist(),
                          on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  np.testing.assert_array_equal(g['sprites'], np.array(sprites))
  # float64 registers at 0 ulp: slope and accumulator, every frame
  np.testing.assert_array_equal(g['floats'].view(np.int64), np.array(floats).view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize('name', NAMES)
def test_facade_apprehend_golden(name):
  """B = 1 facade: the twin's BallSprite draws from the global `random` exactly as
  upstream, one Engine per episode; the device only integrates."""
  from pycolab_b200.games import apprehend
  g = gc.load(name)
  art = tj.u8_to_art(g['art'])
  sprites = []
  random.seed(int(g['random_seed'][0]))
  got = tj.run_trajectory(lambda: apprehend.make_game(art), g['actions'].tolist(),
                          on_frame=lambda env, out: sprites.append(_rows(env)))
  tj.assert_same_trajectory(g, got, name)
  np.testing.assert_array_equal(g['sprites'], np.array(sprites))


@pytest.mark.gpu
def test_batched_apprehend_device_rng_vs_oracle():
  """Auto-resetting batch: env e's slopes come from random.Random(seed + e), drawn by
  the kernel at every restart; boards, rewards, float registers bit-exact."""
  import torch
  from pycolab_b200 import _lib, batched
  from pycolab_b200.games import apprehend
  art = apprehend.GAME_ART
  B, T, seed = 21, 160, 40
  eng = batched.BatchedEngine([apprehend.make_game(art)], batch=B, rng_seed=seed)
  assert eng.rng is not None
  rngs = [random.Random(seed + e) for e in range(B)]
  worlds = [ogames.make_apprehend(art, rngs[e]) for e in range(B)]
  outs = [w.its_showtime() for w in worlds]
  res = eng.its_showtime()
  rs = np.random.RandomState(3)
  episodes = 0
  for t in range(T + 1):
    torch.cuda.synchronize()
    boards = res.board.cpu().numpy()
    spr = eng.sprites.cpu().numpy()
    plot = eng.plot.cpu().numpy()
    for e in range(B):
      np.testing.assert_array_equal(boards[e][:, :len(art[0])], outs[e][0],
                                    err_msg='t=%d env=%d' % (t, e))
      want = outs[e][1]
      assert (int(res.has_reward[e]), int(res.reward[e])) == (
          (0, 0) if want is None else (1, int(want))), (t, e)
      assert float(res.discount[e]) == float(outs[e][2])
      assert bool(res.done[e]) == worlds[e].game_over
      ball = worlds[e].things['b']
      dx = np.array([spr[e, 1, _lib.S_AUX0], spr[e, 1, _lib.S_AUX1]], dtype='<i4').view('<f8')[0]
      acc = np.array([plot[e, _lib.P_AUX0], plot[e, _lib.P_AUX1]], dtype='<i4').view('<f8')[0]
      assert dx == ball.aux['dx'] and acc == ball.aux['acc'], (t, e, dx, ball.aux)
    if t == T:
      break
    act = rs.randint(0, 3, size=B).astype(np.int32)
    res = eng.play(torch.from_numpy(act).cuda())
    for e in range(B):
      if worlds[e].game_over:
        episodes += 1
        worlds[e] = ogames.make_apprehend(art, rngs[e])
        outs[e] = worlds[e].its_showtime()
      else:
        outs[e] = worlds[e].play(int(act[e]))
  assert episodes > 2 * B
  assert int(eng.error_codes().abs().max()) == 0


def test_apprehend_lowers_and_validates_on_cpu():
  from pycolab_b200 import _lib, lowering
  from pycolab_b200.games import apprehend
  random.seed(5)
  want_dx = random.Random(5).uniform(-2.499, 2.499) / 9.0
  game = lowering.lower(apprehend.make_game())
  assert game.program == _lib.PROG_APPREHEND and game.sprite_chars == 'Pb'
  assert game.needs_rng and game.rng_kind == 'python'
  words = game.sprites[1, [_lib.S_AUX0, _lib.S_AUX1]].astype('<i4')
  assert words.view('<f8')[0] == want_dx
  import ctypes as C
  lib = _lib.load()
  handle = C.c_void_p()
  spec = game.make_spec(True)
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(handle)) == _lib.OK
  lib.pcl_destroy(handle)
  spec.sprite_confined[0] = 0                     # a catcher that may leave the board
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(handle)) != _lib.OK


def test_reference_apprehend_file_lowers_like_the_twin():
  """The original's examples/apprehend.py, loaded through `compat` with
  random.seed(11), lowered to what this package's twin lowers to."""
  from pycolab_b200 import lowering
  from pycolab_b200.games import apprehend
  random.seed(11)
  rt.check_lowering('apprehend', lowering.lower(apprehend.make_game()))
