"""GPU parity of scrolly_maze_step on the 64 x 64 board of the generated levels.

That board runs its own instantiation of the step kernel (shape fixed at compile
time, scrolly_maze.cu); the paths a throughput run rarely or never takes are
checked here against the oracle: a ragged last block, quit and out-of-range
actions, long walks with coin pick-ups, masked resets, frozen envs without
auto-reset and the attached cropper.  Bit-exact boards, rewards, discounts, done
flags and curtains.
"""

import numpy as np
import pytest

from oracle import games as ogames

pytestmark = pytest.mark.gpu


def _arts(n, seed0=300):
  from pycolab_b200 import levels
  return [levels.scrolly_maze_level(seed0 + i) for i in range(n)]


def _oracle(arts, e):
  a = arts[e % len(arts)]
  return ogames.make_scrolly_maze(a[0], a[1], '+', a[2])


def _lockstep_with_curtains(arts, actions, auto_reset=True):
  """Step B envs (env e on level e % len(arts)) and B oracle worlds in lockstep;
  returns (engine, number of coins collected)."""
  import torch
  from pycolab_b200 import batched
  from pycolab_b200.games import scrolly_maze
  T, B = actions.shape
  eng = batched.BatchedEngine([scrolly_maze.make_game(*a) for a in arts], batch=B,
                              auto_reset=auto_reset)
  worlds = [_oracle(arts, e) for e in range(B)]
  outs = [w.its_showtime() for w in worlds]
  res = eng.its_showtime()
  acts = torch.from_numpy(actions.astype(np.int32)).cuda()
  collected = 0
  for t in range(T + 1):
    torch.cuda.synchronize()
    boards = res.board.cpu().numpy()
    reward, has = res.reward.cpu().numpy(), res.has_reward.cpu().numpy()
    disc, done = res.discount.cpu().numpy(), res.done.cpu().numpy()
    walls = eng.curtain('#').cpu().numpy()
    coins = eng.curtain('@').cpu().numpy()
    for e in range(B):
      np.testing.assert_array_equal(boards[e], outs[e][0], err_msg='t=%d env=%d' % (t, e))
      want_r = outs[e][1]
      assert (int(has[e]), int(reward[e])) == (
          (0, 0) if want_r is None else (1, int(want_r))), (t, e)
      assert float(disc[e]) == float(outs[e][2]), (t, e)
      assert bool(done[e]) == worlds[e].game_over, (t, e)
      np.testing.assert_array_equal(walls[e], worlds[e].things['#'].curtain,
                                    err_msg='# curtain t=%d env=%d' % (t, e))
      np.testing.assert_array_equal(coins[e], worlds[e].things['@'].curtain,
                                    err_msg='@ curtain t=%d env=%d' % (t, e))
      collected += int(t > 0 and want_r is not None and int(want_r) == 100)
    if t == T:
      break
    res = eng.play(acts[t])
    for e in range(B):
      if worlds[e].game_over:
        if auto_reset:
          worlds[e] = _oracle(arts, e)
          outs[e] = worlds[e].its_showtime()
      else:
        outs[e] = worlds[e].play(int(actions[t, e]))
  assert int(eng.error_codes().max()) == 0
  return eng, collected


@pytest.mark.parametrize('B', [7, 13])
def test_scrolly64_ragged_batch_quit_and_out_of_range_actions(B):
  """B not a multiple of the 4 envs of a block; quits (5) end episodes that
  auto-reset, and actions outside 0..5 move nothing."""
  rs = np.random.RandomState(500 + B)
  actions = rs.choice([0, 1, 2, 3, 4], size=(160, B), p=[.3, .15, .3, .15, .1])
  odd = rs.random_sample(actions.shape)
  actions[odd < 0.02] = 5
  actions[(odd >= 0.02) & (odd < 0.06)] = rs.choice([6, 9, 100, -1, -7], size=int(
      ((odd >= 0.02) & (odd < 0.06)).sum()))
  _lockstep_with_curtains(_arts(3), actions)


def test_scrolly64_long_walks_collect_coins():
  """Runs of one direction: coin pick-ups (the coin window is staged before the
  pick-up and patched in shared memory), curtains compared every step."""
  rs = np.random.RandomState(62)
  actions = np.repeat(rs.randint(0, 4, size=(51, 12)), 6, axis=0)[:300]
  actions[rs.random_sample(actions.shape) < 0.05] = 4
  _, collected = _lockstep_with_curtains(_arts(2, seed0=330), actions)
  assert collected > 0


def test_scrolly64_masked_reset():
  import torch
  from pycolab_b200 import batched
  from pycolab_b200.games import scrolly_maze
  art = _arts(1)[0]
  eng = batched.BatchedEngine([scrolly_maze.make_game(*art)], batch=6, auto_reset=False)
  assert eng.board.shape[1:] == (64, 64)
  first = eng.its_showtime().board.clone()
  rs = np.random.RandomState(0)
  for _ in range(25):
    eng.play(torch.from_numpy(rs.randint(0, 4, size=6).astype(np.int32)).cuda())
  before = eng.board.clone()
  frames = eng.frames().clone()
  mask = torch.tensor([1, 0, 0, 1, 0, 0], dtype=torch.uint8, device='cuda')
  eng.reset(mask)
  torch.cuda.synchronize()
  assert bool((eng.board[[0, 3]] == first[[0, 3]]).all())
  assert bool((eng.board[[1, 2, 4, 5]] == before[[1, 2, 4, 5]]).all())
  assert eng.frames().tolist() == [0, int(frames[1]), int(frames[2]), 0, int(frames[4]),
                                   int(frames[5])]


def test_scrolly64_frozen_without_auto_reset():
  """Envs that quit stay frozen; the others keep matching the oracle."""
  rs = np.random.RandomState(62)
  actions = rs.choice([0, 1, 2, 3, 4], size=(60, 5), p=[.3, .15, .3, .15, .1])
  actions[10, 0] = 5
  actions[25, 3] = 5
  eng, _ = _lockstep_with_curtains(_arts(2, seed0=340), actions, auto_reset=False)
  assert eng.done.tolist()[0] == 1 and eng.done.tolist()[3] == 1
  assert eng.frames().tolist()[0] == 11 and eng.frames().tolist()[3] == 26


def test_scrolly64_attached_cropper():
  """The cropper as the step kernel's epilogue on the 64 x 64 instantiation, against
  the oracle's ScrollingCrop and the stand-alone crop kernel, through auto-resets."""
  import torch
  from oracle import engine_model as em
  from pycolab_b200 import batched
  from pycolab_b200.games import scrolly_maze
  arts = _arts(2, seed0=360)
  B, T = 10, 100
  eng = batched.BatchedEngine([scrolly_maze.make_game(*a) for a in arts], batch=B)
  spec = batched.scrolling_crop_spec(9, 9, 0, pad_char=' ', scroll_margins=(None, None))
  view = eng.attach_cropper(spec)
  assert eng._attached[3], 'the scrolly program runs the cropper inside the step kernel'
  twin_state = eng.new_crop_state()
  worlds = [_oracle(arts, e) for e in range(B)]
  crops = [em.ScrollingCrop(9, 9, ['P'], pad_char=' ', scroll_margins=(None, None))
           for _ in range(B)]
  outs = []
  for w, c in zip(worlds, crops):
    c.set_engine(w)
    outs.append(w.its_showtime())
  eng.its_showtime()
  rs = np.random.RandomState(63)
  actions = rs.choice([0, 1, 2, 3, 4, 5], size=(T, B), p=[.3, .15, .3, .15, .08, .02])
  for t in range(T + 1):
    got = view.cpu().numpy()
    twin = eng.crop(spec, state=twin_state).cpu().numpy()
    np.testing.assert_array_equal(got, twin)
    for e in range(B):
      np.testing.assert_array_equal(got[e], crops[e].crop(outs[e][0]),
                                    err_msg='t=%d env=%d' % (t, e))
    if t == T:
      break
    eng.play(torch.from_numpy(actions[t].astype(np.int32)).cuda())
    for e in range(B):
      if worlds[e].game_over:
        worlds[e] = _oracle(arts, e)
        crops[e].set_engine(worlds[e])
        outs[e] = worlds[e].its_showtime()
      else:
        outs[e] = worlds[e].play(int(actions[t, e]))
