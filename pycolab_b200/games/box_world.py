"""Box-World set-up (reference `pycolab/examples/research/box_world/box_world.py`).

The relational-reasoning benchmark: a room of `grid_size` x `grid_size` cells walled
by '#', keys ('a'..'t'), locks ('A'..'T') and a gem ('*').  A key sits with the lock
it is boxed in on its right; the player ('.') carries one key at a time, shown in
the top-left corner of the board.  Every call of `make_game` draws a new puzzle:
a chain of boxes from a loose key to the gem, plus forward and backward distractor
branches whose locks end the episode with -1.

Set-up only; per-step logic is csrc/box_world.cu.  `make_game` draws from the
`RandomState` exactly what the original does (box_world.py:274-445), so the same
seed gives the same level.
"""

import string

import numpy as np

from pycolab_b200 import ascii_art
from pycolab_b200 import things as plab_things
from pycolab_b200.prefab_parts import sprites as prefab_sprites

GEM = '*'
PLAYER = '.'
BACKGROUND = ' '
BORDER = '#'

MAX_NUM_KEYS = 20
KEYS = list(string.ascii_lowercase[:MAX_NUM_KEYS])
LOCKS = list(string.ascii_uppercase[:MAX_NUM_KEYS])

REWARD_GOAL = 10.
REWARD_STEP = 0.
REWARD_OPEN_CORRECT = 1.
REWARD_OPEN_WRONG = -1.

WALL_WIDTH = 1
MAX_PLACEMENT_TRIES = 200
MAX_GENERATION_TRIES = 200

ACTION_NORTH, ACTION_SOUTH, ACTION_WEST, ACTION_EAST = 0, 1, 2, 3
ACTION_DELAY = -1
ACTION_MAP = {ACTION_NORTH: (-1, 0), ACTION_SOUTH: (1, 0), ACTION_WEST: (0, -1),
              ACTION_EAST: (0, 1)}


def _sample_problem(rand, solution_lengths, num_forwards, num_backwards, branch_length):
  """box_world.py:274-306: the (lock id, key id) of every box; ids index a shuffled
  colour table, lock 0 = no lock, key -1 = the gem.  Box i > solution_length is a
  distractor."""
  solution_length = rand.choice(solution_lengths)
  num_forward = rand.choice(num_forwards)
  num_backward = rand.choice(num_backwards)
  # the path: box 0 holds the loose key 1, box j opens with key j, the last holds the gem
  boxes = [(j, j + 1) for j in range(solution_length)] + [(solution_length, -1)]
  for _ in range(num_forward):                   # branches off a key of the path
    lock = rand.choice(range(1, solution_length + 1))
    for _ in range(branch_length):
      key = None
      while key is None or key == lock:
        key = rand.choice(range(solution_length + 1, MAX_NUM_KEYS))
      boxes.append((lock, key))
      lock = key
  for _ in range(num_backward):                  # a path key locked behind a spare colour
    key = rand.choice(range(1, solution_length + 1))
    lock = rand.choice(range(solution_length + 1, MAX_NUM_KEYS))
    boxes.append((lock, key))
  return int(solution_length), boxes


def _room_for_box(art, x, y):
  """The 3 x 3 square around (y, x) and the column right of it are all background."""
  return (np.all(art[y - 1:y + 2, x - 1:x + 2] == BACKGROUND) and
          np.all(art[y - 1:y + 2, x + 2] == BACKGROUND))


def _draw_level(rand, grid_size, solution_length, num_forward, num_backward, branch_length):
  """One attempt of box_world.py:319-396: (art rows, distractor lock cells (x, y),
  player (x, y)), or None when MAX_PLACEMENT_TRIES ran out."""
  path_length, boxes = _sample_problem(rand, solution_length, num_forward, num_backward,
                                       branch_length)
  colours = list(zip(KEYS, LOCKS))
  rand.shuffle(colours)
  size = grid_size + 2 * WALL_WIDTH
  art = np.full((size, size), BACKGROUND, dtype='<U1')
  art[[0, -1], :] = BORDER
  art[:, [0, -1]] = BORDER
  distractors = []
  misses = 0
  for i, (lock, key) in enumerate(boxes):
    while True:
      if misses > MAX_PLACEMENT_TRIES:
        return None
      x = rand.randint(0, grid_size - 3) + WALL_WIDTH
      y = rand.randint(1, grid_size - 1) + WALL_WIDTH
      if _room_for_box(art, x, y):
        break
      misses += 1
    art[y, x] = GEM if key == -1 else colours[key - 1][0]
    if lock != 0:
      art[y, x + 1] = colours[lock - 1][1]
      if i > path_length:
        distractors.append((x + 1, y))
  while True:
    if misses > MAX_PLACEMENT_TRIES:
      return None
    x = rand.randint(0, grid_size - 1) + WALL_WIDTH
    y = rand.randint(1, grid_size - 1) + WALL_WIDTH
    if art[y, x] == BACKGROUND:
      break
    misses += 1
  art[y, x] = PLAYER
  return [''.join(row) for row in art], distractors, (x, y)


def game_from_art(art, distractors, max_num_steps=120):
  """The Engine of one Box-World level (box_world.py:398-415): `art` with every drape
  character where its curtain is set and '.' at the player; `distractors` the (x, y)
  cells of the distractor locks."""
  grid_size = len(art) - 2 * WALL_WIDTH
  chars = sorted(set(''.join(art)) - {BACKGROUND, BORDER, PLAYER})
  drapes = {}
  for ch in chars:
    klass = GemDrape if ch == GEM else KeyDrape if ch in KEYS else LockDrape
    y, x = [int(v[-1]) for v in np.where(np.array([list(r) for r in art]) == ch)]
    drapes[ch] = ascii_art.Partial(klass, x=x, y=y)
  (py,), (px,) = np.where(np.array([list(r) for r in art]) == PLAYER)
  sprites = {PLAYER: ascii_art.Partial(PlayerSprite, grid_size, int(px), int(py),
                                       list(distractors), max_num_steps)}
  return ascii_art.ascii_art_to_game(
      art=art, what_lies_beneath=BACKGROUND, sprites=sprites, drapes=drapes,
      update_schedule=[PLAYER] + chars, z_order=chars + [PLAYER])


def draw_level(grid_size, solution_length, num_forward, num_backward, branch_length,
               random_state=None):
  """The level `make_game` would build: (art rows, distractor cells, player (x, y))."""
  if random_state is None:
    random_state = np.random.RandomState(None)
  for _ in range(MAX_GENERATION_TRIES):
    level = _draw_level(random_state, grid_size, solution_length, num_forward,
                        num_backward, branch_length)
    if level is not None:
      return level
  raise RuntimeError('Could not generate game in MAX_GENERATION_TRIES tries.')


def make_game(grid_size, solution_length, num_forward, num_backward, branch_length,
              random_state=None, max_num_steps=120):
  """box_world.py:418-445: a new random level; `solution_length`, `num_forward` and
  `num_backward` are the sets each count is drawn from."""
  art, distractors, _ = draw_level(grid_size, solution_length, num_forward, num_backward,
                                   branch_length, random_state)
  return game_from_art(art, distractors, max_num_steps)


class PlayerSprite(prefab_sprites.MazeWalker):
  """Moves N / S / W / E into free cells, opens locks with the key held, takes loose
  keys and the gem; the episode ends after max_num_steps + 1 moves (:127-202)."""

  def __init__(self, corner, position, character, grid_size, x, y, distractors,
               max_num_steps):
    super(PlayerSprite, self).__init__(
        corner, [y, x], character, impassable=BORDER, confined_to_board=True)
    self.distractors = distractors
    self._max_num_steps = max_num_steps
    self._step_counter = 0

  def update(self, actions, board, layers, backdrop, things, the_plot):
    raise NotImplementedError('runs on the device: csrc/box_world.cu')


class BoxThing(plab_things.Drape):
  """A key, lock or gem drape; its cell is also set from (x, y) (:205-229)."""

  def __init__(self, curtain, character, x, y):
    super(BoxThing, self).__init__(curtain, character)
    self.curtain[y][x] = True

  def is_locked_at(self, things, position):
    raise NotImplementedError('runs on the device: csrc/box_world.cu')

  def where_player_over_me(self, the_plot):
    raise NotImplementedError('runs on the device: csrc/box_world.cu')


class GemDrape(BoxThing):
  """+10 and the end of the episode for reaching it (:232-238)."""

  def update(self, actions, board, layers, backdrop, things, the_plot):
    raise NotImplementedError('runs on the device: csrc/box_world.cu')


class KeyDrape(BoxThing):
  """Picked up into the inventory cell (0, 0), dropping the key held (:241-251)."""

  def update(self, actions, board, layers, backdrop, things, the_plot):
    raise NotImplementedError('runs on the device: csrc/box_world.cu')


class LockDrape(BoxThing):
  """Opened by the key of its colour, which it uses up: +1, or -1 and the end of the
  episode for a distractor (:254-271)."""

  def __init__(self, curtain, character, x, y):
    super(LockDrape, self).__init__(curtain, character, x, y)
    self.key_that_opens = KEYS[LOCKS.index(self.character)]

  def update(self, actions, board, layers, backdrop, things, the_plot):
    raise NotImplementedError('runs on the device: csrc/box_world.cu')
