#!/usr/bin/env python
"""Exercise every kernel of libpcl.so at small batch for compute-sanitizer.

    compute-sanitizer --tool memcheck  python tools/sanitize.py
    compute-sanitizer --tool racecheck python tools/sanitize.py
    compute-sanitizer --tool memcheck  python tools/sanitize.py box_world   # that family alone

Small batches (ragged last blocks, the 64 x 64 board, boards that are not multiples of 16 columns,
auto-resets inside the run) so that out-of-bounds accesses and shared-memory
hazards would show.  Prints one line per kernel family; the sanitizer's summary
goes to profiles/ (SURVEY.md §5).
"""

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
  import torch
  from pycolab_b200 import batched, dist as pdist, levels, lowering
  from pycolab_b200.games import (aperture, better_scrolly_maze, extraterrestrial_marauders,
                                  apprehend, fixtures, fluvial_natation, hello_world, ordeal,
                                  shockwave,
                                  scrolly_maze, warehouse_manager)
  from pycolab_b200.games.classics import chain_walk, cliff_walk, four_rooms
  rs = np.random.RandomState(0)
  only = sys.argv[1] if len(sys.argv) > 1 else None     # e.g. `box_world`: that family alone

  def run(name, games, B, n_actions, steps=12, **kw):
    eng = batched.BatchedEngine(games, batch=B, **kw)
    eng.its_showtime()
    for _ in range(steps):
      a = rs.randint(0, n_actions, size=B * eng.actions_per_env).astype(np.int32)
      if eng.game.program == 4:                       # fixture rows: motions + no directives
        a = a.reshape(B, eng.actions_per_env)
        a[:, -8:] = 0
        a[:, :-8] %= 9
      eng.play(torch.from_numpy(a.reshape(-1)).cuda())
    torch.cuda.synchronize()
    assert int(eng.error_codes().abs().max()) in (0, 1, 2), name
    print('ok %-28s B=%d launches=%d' % (name, B, eng.launch_count()))
    return eng

  from pycolab_b200.games import box_world
  pool = [box_world.make_game(12, (1, 2, 3, 4), (0, 1, 2, 3, 4), (0,), 1,
                              random_state=np.random.RandomState(s), max_num_steps=6)
          for s in range(5)]
  run('box_world_step (rotation)', pool, 7, 8, steps=40, cycle_levels=True)
  big = [box_world.make_game(30, (1, 2), (0, 1), (0,), 1, random_state=np.random.RandomState(s),
                             max_num_steps=6) for s in range(3)]
  run('box_world_step 32x32', big, 5, 8, steps=30, cycle_levels=True)
  if only == 'box_world':
    print('done')
    return
  arts = [levels.scrolly_maze_level(5 + i, world_shape=(65, 65), board_shape=(20, 37))
          for i in range(2)]
  eng = run('scrolly_maze_step', [scrolly_maze.make_game(*a) for a in arts], 7, 6)
  spec = batched.scrolling_crop_spec(9, 9, 0, pad_char=' ', scroll_margins=(None, None))
  eng.crop(spec)
  eng.crop(spec, state=eng.new_crop_state())
  eng.unoccluded_layers()
  eng.curtain('#'), eng.curtain('@')
  eng.to_feature_array('P#@ ')
  eng.repaint({'#': '%'})
  fused = pdist.FusedHandoff(eng, spec, eng.batch)
  fused.gather(); fused.gather()
  packed = torch.zeros((eng.batch, pdist.handoff_record_bytes(81)), dtype=torch.uint8, device='cuda')
  eng.pack_handoff(eng.crop(spec), packed)
  torch.cuda.synchronize()
  print('ok crop / layers / export / observe / handoff kernels')
  wide = levels.scrolly_maze_level(9, world_shape=(41, 161), board_shape=(12, 100))
  run('scrolly_maze_step W=100', [scrolly_maze.make_game(*wide)], 5, 5)
  big = [levels.scrolly_maze_level(11 + i) for i in range(2)]        # the fixed-shape instantiation
  eng = run('scrolly_maze_step 64x64', [scrolly_maze.make_game(*a) for a in big], 7, 6)
  eng.attach_cropper(spec)
  for _ in range(6):
    eng.play(torch.from_numpy(rs.randint(0, 6, size=7).astype(np.int32)).cuda())
  torch.cuda.synchronize()
  print('ok scrolly_maze_step 64x64 + attached cropper')
  run('warehouse_step', [warehouse_manager.make_game(
      levels.warehouse_level(3, shape=(14, 21), num_boxes=4, num_goals=5))], 9, 6)
  run('marauders_step', [extraterrestrial_marauders.make_game(levels.marauders_level())], 6, 4,
      steps=40)
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  import golden_cases as gc
  import trajectory as tj
  run('better_scrolly_step',
      [better_scrolly_maze.make_game(tj.u8_to_art(gc.load('better_stock_L1')['art']))], 5, 6)
  for mod in (four_rooms, cliff_walk, chain_walk):
    run('classics_step ' + mod.__name__.rsplit('.', 1)[-1], [mod.make_game()], 5, 4)
  run('classics_step fluvial', [fluvial_natation.make_game()], 5, 3)
  run('aperture_step', [aperture.make_game(levels.aperture_level())], 5, 9)
  for mk in (ordeal.make_castle, ordeal.make_cavern, ordeal.make_kansas):
    g = mk()
    g.the_plot.this_chapter = mk.__name__[5:]
    run('ordeal_step ' + mk.__name__[5:], [g], 5, 5)
  run('hello_step', [hello_world.make_game()], 5, 6)
  run('apprehend_step (device RNG)', [apprehend.make_game()], 5, 3, steps=30)
  run('shockwave_step', [shockwave.make_game(0), shockwave.make_game(levels.shockwave_level(3, 9, 33))][:1], 5, 5, steps=40)
  run('shockwave_step 9x33', [shockwave.make_game(levels.shockwave_level(3, 9, 33))], 6, 5, steps=40)
  pattern = rs.random_sample((17, 23)) < 0.2
  fx = fixtures.make_game(['           ', '   P       ', '      q    ', '           ',
                           '           ', '           '], ' ',
                          {'P': dict(impassable='#', egocentric=True, group='one'),
                           'q': dict(impassable='@', egocentric=True, group='two')},
                          {'#': dict(pattern=pattern, corner=(2, 3), margins=(2, 3), group='one'),
                           '@': dict(pattern=~pattern, corner=(1, 1), margins=None, group='two')},
                          update_schedule=[['#', '@'], ['P', 'q']], z_order='@#Pq')
  run('fixture_step (2 scrolling groups)', [fx], 5, 9)
  print('done')


if __name__ == '__main__':
  main()
