"""Oracle restatement of Box-World (examples/research/box_world/box_world.py:127-415)
in the register-struct style of `oracle.games`.  TEST INFRASTRUCTURE ONLY.

`make_box_world` builds an `engine_model.World` from a generated level the way
ascii_art_to_game + box_world.py:398-415 do; `box_world_program(world, char, actions)`
is the `update()` of the entity that paints `char`, written from the original's
rules (including `the_plot['over_this']`, which is never cleared) rather than from
the device kernel's shortcuts.
"""

import numpy as np

from oracle import engine_model as em
from oracle.games import mask_position, split_art


# ==========================================================================
# box_world (examples/research/box_world/box_world.py:127-271): keys, locks and a gem
# in a walled room; one update group [player] + sorted(drapes), so every entity reads
# the board of the previous step's final render, and the inventory is its cell (0, 0).
# ==========================================================================

BOX_KEYS = 'abcdefghijklmnopqrst'
BOX_LOCKS = 'ABCDEFGHIJKLMNOPQRST'
_BOX_MOTION = {0: em.M_N, 1: em.M_S, 2: em.M_W, 3: em.M_E}          # ACTION_MAP, :119-124


def make_box_world(art, distractors, max_num_steps=120):
  """box_world.py:398-415 over a generated level: `art` rows with '.' at the player,
  `distractors` the (x, y) cells of the distractor locks (:375-376)."""
  chars = sorted(set(''.join(art)) - {' ', '#', '.'})
  backdrop, masks = split_art(art, chars + ['.'], ' ')
  shape = backdrop.shape
  player = em.Walker('.', shape, mask_position(masks['.']), impassable='#',
                     confined=True)                                  # :148-149
  player.aux.update(steps=0, max_steps=int(max_num_steps),
                    distractors=[(int(x), int(y)) for x, y in distractors])
  things = {'.': player}
  for ch in chars:
    things[ch] = em.PlainDrape(ch, masks[ch])
  return em.World(shape[0], shape[1], backdrop, things, z_order=chars + ['.'],
                  groups=[['.'] + chars], program=box_world_program)


def _box_over_me(world, ch):
  """BoxThing.where_player_over_me, :221-229: the cell of the_plot['over_this'] when
  it names `ch` and `ch` still covers it.  The entry is never cleared."""
  over = world.plot.store.get('over_this')
  if over and over[0] == ch and world.things[ch].curtain[over[1]]:
    return over[1]
  return None


def box_world_program(world, ch, actions):
  plot, board, th = world.plot, world.board, world.things
  if ch == '.':                                   # PlayerSprite.update :163-202
    if actions not in _BOX_MOTION:
      return
    pl = th['.']
    plot.add_reward(0.0)                          # REWARD_STEP
    dr, dc = em.MOTIONS[_BOX_MOTION[actions]]
    tr, tc = pl.row + dr, pl.col + dc
    target = chr(board[tr, tc])
    target = None if target == '#' else target    # _in_direction
    thing = th.get(target) if target is not None else None
    held = chr(board[0, 0])
    if thing is None:
      em.walker_move(pl, board, plot, _BOX_MOTION[actions])
    else:
      is_lock = target in BOX_LOCKS
      if is_lock and held == BOX_KEYS[BOX_LOCKS.index(target)]:
        em.walker_move(pl, board, plot, _BOX_MOTION[actions])
      locked = any(c in BOX_LOCKS and th[c].curtain[tr, tc + 1] for c in th)   # :212-219
      if not is_lock and not locked:
        em.walker_move(pl, board, plot, _BOX_MOTION[actions])
    pl.aux['steps'] += 1
    if pl.aux['steps'] > pl.aux['max_steps']:
      plot.terminate_episode()
    if thing is not None:
      plot.store['over_this'] = (target, pl.position)
    return
  where = _box_over_me(world, ch)
  if where is None:
    return
  ent = th[ch]
  if ch == '*':                                   # GemDrape :235-238
    plot.add_reward(10.0)
    plot.terminate_episode()
  elif ch in BOX_KEYS:                            # KeyDrape :244-251
    held = chr(board[0, 0])
    if held in BOX_KEYS:
      th[held].curtain[0, 0] = False
    ent.curtain[where] = False
    ent.curtain[0, 0] = True
  else:                                           # LockDrape :261-271
    ent.curtain[where] = False
    th[chr(board[0, 0])].curtain[0, 0] = False
    if (where[1], where[0]) in th['.'].aux['distractors']:
      plot.add_reward(-1.0)
      plot.terminate_episode()
    else:
      plot.add_reward(1.0)


def box_world_plane(world):
  """The cell plane the device keeps (pcl.h PCL_PROG_BOX_WORLD): u8 [rows, cols], the
  character of the drape covering each cell, bit 7 on distractor lock cells."""
  plane = np.zeros((world.rows, world.cols), dtype=np.uint8)
  for ch, ent in world.things.items():
    if not ent.is_sprite:
      assert not np.any(plane[ent.curtain]), 'drapes overlap'
      plane[ent.curtain] = ord(ch)
  for x, y in world.things['.'].aux['distractors']:
    if chr(plane[y, x]) in BOX_LOCKS:
      plane[y, x] |= 0x80
  return plane
