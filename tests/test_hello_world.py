"""examples/hello_world.py (SURVEY.md §8f-4): plain wrapping Sprites + a rolling
Drape.  Goldens are the reference's own trajectories (tests/golden/hello_stock_*);
CPU: the oracle; GPU: the facade Engine (B = 1) and a batched lockstep."""

import os

import numpy as np
import pytest

import golden_cases as gc
import reference_trace as rt
import trajectory as tj
from oracle import games as ogames

NAMES = gc.names('hello_')


def _rows(env, chars='1234'):
  out = []
  for ch in chars:
    s = env.things[ch]
    out.append([int(s.position[0]), int(s.position[1]), int(bool(s.visible)),
                int(s.position[0]), int(s.position[1])])
  return out


@pytest.mark.parametrize('name', NAMES)
def test_oracle_hello_matches_reference_golden(name):
  g = gc.load(name)
  art = tj.u8_to_art(g['art'])
  sprites, curtains = [], []

  def on_frame(env, out):
    sprites.append(_rows(env))
    curtains.append(env.things['@'].curtain.copy())
  got = tj.run_trajectory(lambda: ogames.make_hello(art), g['actions'].tolist(),
                          on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  np.testing.assert_array_equal(g['sprites'], np.array(sprites))
  np.testing.assert_array_equal(g['curtains'].astype(bool), np.stack(curtains))


@pytest.mark.gpu
@pytest.mark.parametrize('name', NAMES)
def test_facade_hello_golden(name):
  from pycolab_b200.games import hello_world
  g = gc.load(name)
  art = tj.u8_to_art(g['art'])
  sprites, curtains = [], []

  def on_frame(env, out):
    sprites.append(_rows(env))
    curtains.append(env.things['@'].curtain.copy())
  got = tj.run_trajectory(lambda: hello_world.make_game(art), g['actions'].tolist(),
                          on_frame=on_frame)
  tj.assert_same_trajectory(g, got, name)
  np.testing.assert_array_equal(g['sprites'], np.array(sprites))
  np.testing.assert_array_equal(g['curtains'].astype(bool), np.stack(curtains))


@pytest.mark.gpu
def test_batched_hello_vs_oracle():
  import torch
  from pycolab_b200 import batched
  from pycolab_b200.games import hello_world
  art = hello_world.HELLO_ART
  B, T = 19, 200
  eng = batched.BatchedEngine([hello_world.make_game(art)], batch=B)
  worlds = [ogames.make_hello(art) for _ in range(B)]
  outs = [w.its_showtime() for w in worlds]
  res = eng.its_showtime()
  rs = np.random.RandomState(8)
  for t in range(T + 1):
    torch.cuda.synchronize()
    boards = res.board.cpu().numpy()
    cur = eng.curtain('@').cpu().numpy()
    for e in range(B):
      np.testing.assert_array_equal(boards[e], outs[e][0], err_msg='t=%d env=%d' % (t, e))
      np.testing.assert_array_equal(cur[e], worlds[e].things['@'].curtain)
      want = outs[e][1]
      assert (int(res.has_reward[e]), int(res.reward[e])) == (
          (0, 0) if want is None else (1, int(want))), (t, e)
      assert float(res.discount[e]) == float(outs[e][2]) and bool(res.done[e]) == worlds[e].game_over
    if t == T:
      break
    act = rs.choice([0, 1, 2, 3, 4, 5], size=B, p=[.23, .23, .23, .23, .03, .05]).astype(np.int32)
    res = eng.play(torch.from_numpy(act).cuda())
    for e in range(B):
      if worlds[e].game_over:
        worlds[e] = ogames.make_hello(art)
        outs[e] = worlds[e].its_showtime()
      else:
        outs[e] = worlds[e].play(int(act[e]))
  assert int(eng.error_codes().abs().max()) == 0


def test_reference_hello_world_file_lowers_like_the_twin():
  """The original's examples/hello_world.py, loaded through `compat`, lowered to
  what this package's twin lowers to."""
  from pycolab_b200 import lowering
  from pycolab_b200.games import hello_world
  with rt.sorted_default_schedule():
    game = hello_world.make_game()
  rt.check_lowering('hello_world', lowering.lower(game))
