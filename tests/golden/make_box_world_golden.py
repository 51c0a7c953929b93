"""Generate the Box-World golden fixtures from the unmodified original.

Run with PYCOLAB_UPSTREAM naming an upstream pycolab checkout:

    python tests/golden/make_box_world_golden.py

Writes, next to this file:
  box_world_levels.npz      the levels the original's make_game draws for the seeds of
                            tests/box_world_cases.LEVEL_SEEDS: art, distractor cells,
                            player cell, per parameter set;
  box_world_*.npz           the tapes of tests/box_world_cases.TAPES, played on the
                            original with the scripted or random policy: per frame the
                            board, reward, discount, game_over, the player's row, column
                            and step counter, and every drape's curtain as one plane of
                            characters;
  box_world_lowerings.json  how the original's file, loaded through pycolab_b200.compat,
                            lowers for a few seeds (tests/reference_trace.lowering_digest).
"""

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import box_world_cases as cases
import refdriver

REL_PATH = os.path.join('pycolab', 'examples', 'research', 'box_world', 'box_world.py')
LOWERING_SEEDS = (0, 1, 2, 3)


def lowerings():
  """Digests of the original's file lowered through compat (before the upstream
  package itself is imported: both answer to the name `pycolab`)."""
  from pycolab_b200 import compat, lowering
  import reference_trace
  module = compat.load_example(os.path.join(refdriver.REFERENCE_ROOT, REL_PATH))
  out = {}
  for seed in LOWERING_SEEDS:
    game = module.make_game(*cases.PARAMS['default'], random_state=np.random.RandomState(seed))
    out['box_world_%d' % seed] = reference_trace.lowering_digest(lowering.lower(game))
  compat.uninstall()
  path = os.path.join(HERE, 'box_world_lowerings.json')
  with open(path, 'w') as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write('\n')
  print('box_world_lowerings.json', out)


def upstream():
  if refdriver.REFERENCE_ROOT not in sys.path:
    sys.path.insert(0, refdriver.REFERENCE_ROOT)
  from pycolab.examples.research.box_world import box_world
  return box_world


def board_of(obs):
  return np.array(obs.board, dtype=np.uint8)


def plane_of(game):
  """Every drape's curtain as one u8 plane of characters (asserting no overlap)."""
  plane = None
  for ch, ent in game.things.items():
    if ch == '.':
      continue
    if plane is None:
      plane = np.zeros(ent.curtain.shape, dtype=np.uint8)
    assert not np.any(plane[ent.curtain]), 'drapes overlap'
    plane[ent.curtain] = ord(ch)
  return plane


def levels(bw):
  out = {'params': json.dumps(cases.PARAMS)}
  for name, seeds in cases.LEVEL_SEEDS.items():
    arts, dists, players = [], [], []
    for seed in seeds:
      game = bw.make_game(*cases.PARAMS[name], random_state=np.random.RandomState(seed))
      obs, _, _ = game.its_showtime()
      arts.append(board_of(obs))
      d = np.full((24, 2), -1, dtype=np.int32)
      for i, (x, y) in enumerate(game.things['.'].distractors):
        d[i] = (x, y)
      dists.append(d)
      r, c = game.things['.'].position
      players.append((c, r))
    out[name + '_seeds'] = np.array(list(seeds), dtype=np.int32)
    out[name + '_art'] = np.stack(arts)
    out[name + '_distractors'] = np.stack(dists)
    out[name + '_player'] = np.array(players, dtype=np.int32)
  np.savez_compressed(os.path.join(HERE, 'box_world_levels.npz'), **out)
  print('box_world_levels.npz', {k: v.shape for k, v in out.items() if k != 'params'})


def game_from_art(bw, art, distractors, limit):
  """The original's classes on a given level, assembled as box_world.py:398-415 does."""
  from pycolab import ascii_art
  chars = sorted(set(''.join(art)) - set(' #.'))
  grid = np.array([list(row) for row in art])
  drapes = {}
  for ch in chars:
    klass = bw.GemDrape if ch == '*' else bw.KeyDrape if ch in cases.KEYS else bw.LockDrape
    ys, xs = np.where(grid == ch)
    drapes[ch] = ascii_art.Partial(klass, x=int(xs[-1]), y=int(ys[-1]))
  (py,), (px,) = np.where(grid == '.')
  sprites = {'.': ascii_art.Partial(bw.PlayerSprite, len(art) - 2, int(px), int(py),
                                    list(distractors), limit)}
  return ascii_art.ascii_art_to_game(art=art, what_lies_beneath=' ', sprites=sprites,
                                     drapes=drapes, update_schedule=['.'] + chars,
                                     z_order=chars + ['.'])


def tape(bw, name):
  pset, seed0, steps, policy, epsilon, limit = cases.TAPES[name]
  rng = np.random.RandomState(seed0 + 7)
  rec = {k: [] for k in ('board', 'plane', 'reward', 'has_reward', 'discount', 'game_over',
                         'player', 'action', 'showtime', 'episode')}
  arts, dists, seeds = [], [], []
  game, obs, seed = None, None, seed0
  noop = 0
  for t in range(steps):
    if game is None or game.game_over:
      if pset == 'handmade':
        game = game_from_art(bw, cases.HANDMADE_ART, cases.HANDMADE_DISTRACTORS, limit)
        seeds.append(-1)
      else:
        game = bw.make_game(*cases.PARAMS[pset], random_state=np.random.RandomState(seed),
                            max_num_steps=limit)
        seeds.append(seed)
        seed += 1
      d = np.full((24, 2), -1, dtype=np.int32)
      for i, (x, y) in enumerate(game.things['.'].distractors):
        d[i] = (x, y)
      dists.append(d)
      obs, reward, discount = game.its_showtime()
      arts.append(board_of(obs))
      action, first = -1, True
    else:
      changed = len(rec['plane']) > 1 and not np.array_equal(rec['plane'][-1], rec['plane'][-2])
      if changed and not rec['showtime'][-1] and rng.rand() < 0.5:
        action = cases.NOOP_ACTIONS[noop % 3]      # a no-op right after a pick-up / opening
        noop += 1
      else:
        action = cases.policy_action(board_of(obs), rng, policy, epsilon)
      obs, reward, discount = game.play(action)
      first = False
    pl = game.things['.']
    rec['board'].append(board_of(obs))
    rec['plane'].append(plane_of(game))
    rec['reward'].append(np.nan if reward is None else float(reward))
    rec['has_reward'].append(reward is not None)
    rec['discount'].append(float(discount))
    rec['game_over'].append(bool(game.game_over))
    rec['player'].append((pl.position[0], pl.position[1], pl._step_counter))
    rec['action'].append(action)
    rec['showtime'].append(first)
    rec['episode'].append(len(seeds) - 1)
  out = dict(
      board=np.stack(rec['board']), plane=np.stack(rec['plane']),
      reward=np.array(rec['reward'], dtype=np.float64),
      has_reward=np.array(rec['has_reward'], dtype=np.uint8),
      discount=np.array(rec['discount'], dtype=np.float64),
      game_over=np.array(rec['game_over'], dtype=np.uint8),
      player=np.array(rec['player'], dtype=np.int32),
      action=np.array(rec['action'], dtype=np.int32),
      showtime=np.array(rec['showtime'], dtype=np.uint8),
      episode=np.array(rec['episode'], dtype=np.int32),
      art=np.stack(arts), distractors=np.stack(dists), seeds=np.array(seeds, dtype=np.int32),
      params=json.dumps(cases.PARAMS.get(pset)), max_num_steps=limit)
  np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
  print('%-24s %d frames, %d episodes, events %s' % (
      name, steps, len(seeds), sorted(cases.tape_events(out))))


def main():
  assert refdriver.available(), refdriver.MISSING
  lowerings()
  bw = upstream()
  levels(bw)
  for name in cases.TAPES:
    tape(bw, name)


if __name__ == '__main__':
  main()
