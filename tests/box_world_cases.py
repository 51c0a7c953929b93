"""Box-World test cases: level parameter sets, the scripted policy, the recorded tapes
and the event checks shared by tests/golden/make_box_world_golden.py and
tests/test_box_world.py.

A tape is a run of consecutive episodes on one parameter set: when an episode ends
the next one starts on the level of the next seed.  Frame 0 of every episode is its
its_showtime() frame.
"""

import collections
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

KEYS = 'abcdefghijklmnopqrst'
LOCKS = 'ABCDEFGHIJKLMNOPQRST'
MOVES = ((-1, 0), (1, 0), (0, -1), (0, 1))          # actions 0..3: N S W E
# Besides the four moves: -1 (ACTION_DELAY), 4 and 7 (out of range) are no-ops.
NOOP_ACTIONS = (-1, 4, 7)

# (grid_size, solution_length, num_forward, num_backward, branch_length)
PARAMS = {
    'default': (12, (1, 2, 3, 4), (0, 1, 2, 3, 4), (0,), 1),
    'backward': (12, (1, 2, 3), (0, 1, 2), (1, 2), 2),
    'large': (20, (1, 2, 3, 4), (0, 1, 2, 3, 4), (0,), 1),
}
LEVEL_SEEDS = {'default': range(0, 70), 'backward': range(100, 170), 'large': range(200, 270)}

# name -> (parameter set, first seed, steps, policy, epsilon, max_num_steps)
TAPES = {
    'box_world_scripted_a': ('default', 1000, 400, 'scripted', 0.15, 120),
    'box_world_scripted_b': ('default', 2000, 400, 'scripted', 0.3, 120),
    'box_world_backward': ('backward', 3000, 400, 'scripted', 0.2, 120),
    'box_world_large': ('large', 4000, 400, 'scripted', 0.2, 120),
    'box_world_random': ('default', 5000, 400, 'random', 1.0, 120),
    'box_world_short': ('default', 6000, 300, 'scripted', 0.5, 30),
    'box_world_handmade': ('handmade', 0, 300, 'scripted', 0.1, 120),
}

# A level the generator never draws: two loose keys at once, so that taking the second
# drops the first (a key swap); the lock 'A' boxes the key 'd', the distractor lock
# 'D' the key 'e', and 'C' the gem.  Replayed whole after every episode.
HANDMADE_ART = [
    '##############',
    '#            #',
    '# a  b       #',
    '#            #',
    '#     .      #',
    '#            #',
    '#   cB    eD #',
    '#            #',
    '#   *C       #',
    '#            #',
    '#         dA #',
    '#            #',
    '#            #',
    '##############']
HANDMADE_DISTRACTORS = [(11, 6)]


def policy_action(board, rng, policy, epsilon):
  """An action for `board` (u8 [rows, cols], the last observation).  'random': any of
  the moves and no-ops.  'scripted': with probability 1 - epsilon a step along a
  shortest path to the nearest useful cell (the gem or a key without a lock on its
  right, or the lock that the key held opens), else a random action."""
  if policy == 'random' or rng.rand() < epsilon:
    return int(rng.choice([0, 1, 2, 3, 0, 1, 2, 3] + list(NOOP_ACTIONS)))
  rows, cols = board.shape
  (pr,), (pc,) = np.where(board == ord('.'))
  held = chr(board[0, 0])

  def useful(r, c):
    ch = chr(board[r, c])
    loose = c + 1 < cols and chr(board[r, c + 1]) not in LOCKS
    if ch == '*' or (ch in KEYS and ch != held):
      return loose
    return ch in LOCKS and held == ch.lower()

  first = {(pr, pc): None}
  queue = collections.deque([(pr, pc)])
  while queue:
    r, c = queue.popleft()
    for a, (dr, dc) in enumerate(MOVES):
      nr, nc = r + dr, c + dc
      if (nr, nc) in first or not (0 < nr < rows - 1 and 0 < nc < cols - 1):
        continue
      step = a if first[(r, c)] is None else first[(r, c)]
      if useful(nr, nc):
        return step
      if board[nr, nc] == ord(' '):
        first[(nr, nc)] = step
        queue.append((nr, nc))
  return int(rng.randint(0, 4))


def load_tape(name):
  with np.load(os.path.join(GOLDEN_DIR, name + '.npz')) as z:
    return {k: z[k] for k in z.files}


def tape_events(tape):
  """The events a tape contains, from its recorded frames."""
  ev = set()
  boards, planes, actions = tape['board'], tape['plane'], tape['action']
  reward, over, first = tape['reward'], tape['game_over'], tape['showtime']
  player, limit = tape['player'], int(tape['max_num_steps'])
  for t in range(len(actions)):
    if first[t]:
      continue
    a = int(actions[t])
    if a in NOOP_ACTIONS:
      ev.add('action_%d' % a)
    if reward[t] >= 10.0:
      ev.add('gem')
    if over[t] and reward[t] == -1.0:
      ev.add('distractor')
    if over[t] and int(player[t, 2]) == limit + 1 and reward[t] == 0.0:
      ev.add('timeout')
    if a in NOOP_ACTIONS and not first[t - 1] and not np.array_equal(planes[t - 1],
                                                                      planes[t - 2]):
      ev.add('noop_after_event')                 # the_plot['over_this'] is still set
    held0, held1 = planes[t - 1][0, 0], planes[t][0, 0]
    if held0 and held1 and held0 != held1 and chr(held1) in KEYS:
      ev.add('key_swap')
    if 0 <= a < 4 and tuple(player[t, :2]) == tuple(player[t - 1, :2]):
      r, c = player[t - 1, :2] + np.array(MOVES[a])
      ch = chr(boards[t - 1][r, c])
      locked = chr(boards[t - 1][r, c + 1]) in LOCKS if c + 1 < boards.shape[2] else False
      if ch == '#':
        ev.add('bump_wall')
      elif ch in KEYS and locked:
        ev.add('bump_locked_key')
      elif ch == '*' and locked:
        ev.add('bump_locked_gem')
      elif ch in LOCKS and chr(boards[t - 1][0, 0]) != ch.lower():
        ev.add('bump_lock_without_key')
  for art in tape['art']:
    chars = [chr(v) for v in art.ravel() if chr(v) not in ' #.']
    if len(chars) != len(set(chars)):
      ev.add('duplicate_chars')
  return ev


REQUIRED_EVENTS = {'gem', 'distractor', 'timeout', 'key_swap', 'bump_wall', 'bump_locked_key',
                   'bump_locked_gem', 'bump_lock_without_key', 'action_-1', 'action_4',
                   'action_7', 'duplicate_chars', 'noop_after_event'}
