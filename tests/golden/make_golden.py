"""Generate the golden fixtures in this directory from the REAL reference.

Run with PYCOLAB_UPSTREAM naming an upstream pycolab checkout:

    python tests/golden/make_golden.py

Every .npz written here holds the inputs (level art as uint8 arrays, action
stream, RNG seed, entity configuration as JSON) and the outputs the unmodified
reference produced for them (board per frame, reward, discount, game_over,
sprite registers, crops).  The GPU box has no /root/reference: the `-m gpu`
parity tests and the oracle tests compare against these files.
"""

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import refdriver
import trajectory as tj
from pycolab_b200 import levels


def save(name, **arrays):
  path = os.path.join(HERE, name + '.npz')
  np.savez_compressed(path, **arrays)
  print('%-32s %8.1f KiB' % (name, os.path.getsize(path) / 1024.0))


def sprite_recorder(chars, sink):
  def on_frame(env, out):
    things = env.things
    row = []
    for ch in chars:
      s = things[ch]
      vp = getattr(s, 'virtual_position', s.position)
      row.append([int(s.position[0]), int(s.position[1]), int(bool(s.visible)),
                  int(vp[0]), int(vp[1])])
    sink.append(row)
  return on_frame


def scrolly(name, maze, board, beneath, actions, level=None):
  sprites = []
  if level is not None:
    make = lambda: refdriver.ref_scrolly_maze(None, None, level=level)
  else:
    make = lambda: refdriver.ref_scrolly_maze(maze, board, beneath)
  traj = tj.run_trajectory(make, actions,
                           on_frame=sprite_recorder('Pabc', sprites))
  save(name, maze_art=tj.art_to_u8(maze), board_art=tj.art_to_u8(board),
       beneath=np.array([ord(beneath)], dtype=np.uint8),
       actions=np.array(actions, dtype=np.int32),
       sprites=np.array(sprites, dtype=np.int32), **traj)


def warehouse(name, art, wlb, actions, level=None):
  chars = [c for c in '1234567890' if c in ''.join(art)] + ['P']
  sprites = []
  if level is not None:
    make = lambda: refdriver.ref_warehouse(None, level=level)
  else:
    make = lambda: refdriver.ref_warehouse(art, wlb)
  traj = tj.run_trajectory(make, actions,
                           on_frame=sprite_recorder(chars, sprites))
  wlb_arr = (np.array([[ord(wlb)]], dtype=np.uint8) if isinstance(wlb, str)
             else tj.art_to_u8(wlb))
  save(name, art=tj.art_to_u8(art), what_lies_beneath=wlb_arr,
       sprite_chars=np.frombuffer(''.join(chars).encode(), dtype=np.uint8),
       actions=np.array(actions, dtype=np.int32),
       sprites=np.array(sprites, dtype=np.int32), **traj)


def marauders(name, seed, actions):
  art = refdriver.ref_stock_marauders_art()
  chars = 'Pabcdyz'
  sprites = []
  np.random.seed(seed)            # the reference uses the global NumPy RNG
  traj = tj.run_trajectory(lambda: refdriver.ref_marauders(), actions,
                           on_frame=sprite_recorder(chars, sprites))
  save(name, art=tj.art_to_u8(art), rng_seed=np.array([seed], dtype=np.int64),
       actions=np.array(actions, dtype=np.int32),
       sprites=np.array(sprites, dtype=np.int32), **traj)


def fixture_walkers(name, seed, T=300):
  rs = np.random.RandomState(seed)
  H, W = int(rs.randint(5, 12)), int(rs.randint(5, 14))
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[rs.random_sample((H, W)) < 0.25] = ord('#')
  art[rs.random_sample((H, W)) < 0.1] = ord('%')
  free = np.argwhere(art == ord(' '))
  picks = free[rs.permutation(len(free))[:3]]
  for ch, (r, c) in zip('abc', picks):
    art[r, c] = ord(ch)
  walkers = {
      'a': dict(impassable='#', confined=bool(rs.randint(2))),
      'b': dict(impassable='#%a', confined=bool(rs.randint(2))),
      'c': dict(impassable='', confined=False),
  }
  schedule = [['a'], ['b', 'c']] if rs.randint(2) else [['a', 'b', 'c']]
  z_order = ''.join(rs.permutation(list('abc')))
  art_l = tj.u8_to_art(art)
  motions = rs.randint(0, 9, size=(T, 3)).astype(np.int32)
  sprites = []
  traj = tj.run_trajectory(
      lambda: refdriver.ref_fixture(art_l, ' ', walkers,
                                    update_schedule=schedule, z_order=z_order),
      motions,
      convert_action=lambda m: refdriver.fixture_actions_to_ref(
          {ch: int(v) for ch, v in zip('abc', m)}),
      on_frame=sprite_recorder('abc', sprites))
  cfg = dict(walkers=walkers, scrollys={}, drapes='', schedule=schedule,
             z_order=z_order, what_lies_beneath=' ', action_chars='abc')
  save(name, art=art, config=np.frombuffer(json.dumps(cfg).encode(), np.uint8),
       actions=motions, sprites=np.array(sprites, dtype=np.int32), **traj)


def fixture_scrolly(name, seed, margins, second_ego, T=400):
  rs = np.random.RandomState(1000 + seed)
  PH, PW, H, W = 17, 23, 8, 11
  pattern = rs.random_sample((PH, PW)) < 0.2
  pattern2 = rs.random_sample((PH, PW)) < 0.1
  corner = (int(rs.randint(0, PH - H + 1)), int(rs.randint(0, PW - W + 1)))
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[3, 4] = ord('P')
  art[5, 7] = ord('q')
  art_l = tj.u8_to_art(art)
  walkers = {'P': dict(impassable='#', egocentric=True),
             'q': dict(impassable='#', egocentric=bool(second_ego))}
  scrollys = {'#': dict(pattern=pattern, corner=corner, margins=margins),
              '@': dict(pattern=pattern2, corner=corner, margins=margins)}
  schedule = [['#'], ['P', 'q'], ['@']]
  motions = rs.randint(0, 9, size=(T,)).astype(np.int32)
  sprites, curtains = [], []
  rec = sprite_recorder('Pq', sprites)

  def on_frame(env, out):
    rec(env, out)
    curtains.append(np.stack([env.things['#'].curtain.copy(),
                              env.things['@'].curtain.copy()]))

  env = refdriver.ref_fixture(art_l, ' ', walkers, scrollys,
                              update_schedule=schedule, z_order='@#Pq')
  out = env.its_showtime()
  boards = [tj.board_of(out[0]).copy()]
  on_frame(env, out)
  used = []
  for m in motions:
    try:
      out = env.play(refdriver.fixture_actions_to_ref(int(m)))
    except RuntimeError:
      break                         # reference rejects a (0,0)-clipped order
    used.append(int(m))
    boards.append(tj.board_of(out[0]).copy())
    on_frame(env, out)
  cfg = dict(
      walkers=walkers,
      scrollys={ch: dict(corner=list(corner),
                         margins=None if margins is None else list(margins))
                for ch in '#@'},
      drapes='', schedule=schedule, z_order='@#Pq', what_lies_beneath=' ',
      action_chars='')
  save(name, art=art, config=np.frombuffer(json.dumps(cfg).encode(), np.uint8),
       pattern_hash=pattern.astype(np.uint8), pattern_at=pattern2.astype(np.uint8),
       actions=np.array(used, dtype=np.int32), boards=np.stack(boards),
       sprites=np.array(sprites, dtype=np.int32),
       curtains=np.stack(curtains).astype(np.uint8))


def fixture_groups(name, seed, margins, T=400):
  """Two scrolling groups at once (protocols/scrolling.py:198-241): group 'one' =
  Scrolly '#' + egocentric walker P, group 'two' = Scrolly '@' + egocentric walker q;
  every step each group gets its own random motion, so the two windows scroll
  independently and each walker obeys only its own group's orders."""
  rs = np.random.RandomState(2000 + seed)
  PH, PW, H, W = 17, 23, 8, 11
  pattern = rs.random_sample((PH, PW)) < 0.2
  pattern2 = rs.random_sample((PH, PW)) < 0.1
  corner = (int(rs.randint(0, PH - H + 1)), int(rs.randint(0, PW - W + 1)))
  corner2 = (int(rs.randint(0, PH - H + 1)), int(rs.randint(0, PW - W + 1)))
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[3, 4] = ord('P')
  art[5, 7] = ord('q')
  art_l = tj.u8_to_art(art)
  walkers = {'P': dict(impassable='#', egocentric=True, group='one'),
             'q': dict(impassable='@', egocentric=True, group='two')}
  scrollys = {'#': dict(pattern=pattern, corner=corner, margins=margins, group='one'),
              '@': dict(pattern=pattern2, corner=corner2, margins=margins, group='two')}
  schedule = [['#', '@'], ['P', 'q']]
  motions = rs.randint(0, 9, size=(T, 2)).astype(np.int32)      # (group one, group two)
  sprites, curtains = [], []
  rec = sprite_recorder('Pq', sprites)

  def on_frame(env, out):
    rec(env, out)
    curtains.append(np.stack([env.things['#'].curtain.copy(),
                              env.things['@'].curtain.copy()]))

  env = refdriver.ref_fixture(art_l, ' ', walkers, scrollys,
                              update_schedule=schedule, z_order='@#Pq')
  out = env.its_showtime()
  boards = [tj.board_of(out[0]).copy()]
  on_frame(env, out)
  used = []
  for m1, m2 in motions:
    act = {'#': int(m1), 'P': int(m1), '@': int(m2), 'q': int(m2)}
    try:
      out = env.play(refdriver.fixture_actions_to_ref(act))
    except RuntimeError:
      break                         # reference rejects a (0,0)-clipped order
    used.append([int(m1), int(m2)])
    boards.append(tj.board_of(out[0]).copy())
    on_frame(env, out)
  cfg = dict(
      walkers=walkers,
      scrollys={'#': dict(corner=list(corner), group='one',
                          margins=None if margins is None else list(margins)),
                '@': dict(corner=list(corner2), group='two',
                          margins=None if margins is None else list(margins))},
      drapes='', schedule=schedule, z_order='@#Pq', what_lies_beneath=' ',
      action_chars='', motion_of=dict([('#', 0), ('P', 0), ('@', 1), ('q', 1)]))
  save(name, art=art, config=np.frombuffer(json.dumps(cfg).encode(), np.uint8),
       pattern_hash=pattern.astype(np.uint8), pattern_at=pattern2.astype(np.uint8),
       actions=np.array(used, dtype=np.int32).reshape(-1, 2), boards=np.stack(boards),
       sprites=np.array(sprites, dtype=np.int32),
       curtains=np.stack(curtains).astype(np.uint8))
  print('  %s: %d steps' % (name, len(used)))


def ordeals():
  """examples/ordeal.py through the reference's own Story (cropped observations,
  summed rewards across chapter crossings, discounts, chapter names, has_sword)."""
  import ordeal_cases
  mods = refdriver.ref_storytelling()
  from pycolab.examples import ordeal as ref_ordeal
  for name, actions in sorted(ordeal_cases.scripts().items()):
    chapters, swords = [], []

    def on_frame(env, out):
      chapters.append(str(env.the_plot.this_chapter))
      swords.append(1 if env.the_plot.get('has_sword') else 0)
    traj = tj.run_trajectory(ref_ordeal.make_game, actions, on_frame=on_frame)
    save(name, actions=np.array(actions, dtype=np.int32),
         chapters=np.array(chapters), has_sword=np.array(swords, dtype=np.uint8), **traj)
    print('  %s: %d steps, chapters %s, reward sum %s' % (
        name, len(traj['boards']) - 1, sorted(set(chapters)), traj['reward'].sum()))


def hellos():
  """examples/hello_world.py: stock art, random actions 0-5 (4 quits, 5 is a no-op)."""
  refdriver._import()
  from pycolab.examples import hello_world as ref_hello
  for seed in range(2):
    rs = np.random.RandomState(600 + seed)
    actions = rs.choice([0, 1, 2, 3, 4, 5], size=400, p=[.22, .22, .22, .22, .02, .10]).tolist()
    sprites, curtains = [], []
    rec = sprite_recorder('1234', sprites)

    def on_frame(env, out):
      rec(env, out)
      curtains.append(env.things['@'].curtain.copy())
    traj = tj.run_trajectory(ref_hello.make_game, actions, on_frame=on_frame)
    save('hello_stock_s%d' % seed, art=tj.art_to_u8(ref_hello.HELLO_ART),
         actions=np.array(actions, dtype=np.int32), sprites=np.array(sprites, dtype=np.int32),
         curtains=np.stack(curtains).astype(np.uint8), **traj)


def apprehends():
  """examples/apprehend.py: stock art; `random.seed` fixes the global stream the ball
  sprites draw their slopes from (one draw per episode), actions 0-2 (2 = stay put)."""
  import random
  refdriver._import()
  from pycolab.examples import apprehend as ref_app
  for seed in range(3):
    rs = np.random.RandomState(700 + seed)
    actions = rs.randint(0, 3, size=300).tolist()
    sprites, floats = [], []
    rec = sprite_recorder('Pb', sprites)

    def on_frame(env, out):
      rec(env, out)
      floats.append([env.things['b']._dx, env.things['b']._x_accumulator])
    random.seed(700 + seed)
    traj = tj.run_trajectory(ref_app.make_game, actions, on_frame=on_frame)
    save('apprehend_stock_s%d' % seed, art=tj.art_to_u8(ref_app.GAME_ART),
         actions=np.array(actions, dtype=np.int32), sprites=np.array(sprites, dtype=np.int32),
         floats=np.array(floats, dtype=np.float64), random_seed=np.array([700 + seed]), **traj)
    print('  apprehend_stock_s%d: %d episodes, reward sum %d' % (
        seed, int(traj['game_over'].sum()), int(traj['reward'].sum())))


def shockwaves():
  """examples/shockwave.py: the stock level and two generated ones (12x15, 20x40);
  `np.random.seed` fixes the global stream the impact points come from; actions 0-4
  (4 = none of the keys), biased upwards so that some episodes are won."""
  refdriver._import()
  from pycolab.examples import shockwave as ref_shock
  from pycolab_b200 import levels
  cases = [('stock', ref_shock.LEVELS[0]), ('g12x15', levels.shockwave_level(1, safety_density=0.5)),
           ('g20x40', levels.shockwave_level(2, 20, 40, 0.6))]
  for seed, (tag, art) in enumerate(cases):
    ref_shock.LEVELS.append(art)
    make = lambda: ref_shock.make_game(len(ref_shock.LEVELS) - 1)
    try:
      # pass 1: a climbing policy that looks at the reference env (up when the cell
      # above is free, else sideways; sometimes waits) chooses the actions ...
      rs = np.random.RandomState(800 + seed)
      np.random.seed(800 + seed)
      actions, env = [], make()
      env.its_showtime()
      for _ in range(500):
        if env.game_over:
          env = make()
          env.its_showtime()
          actions.append(int(rs.randint(0, 5)))        # ignored by the protocol
          continue
        r, c = env.things['P'].position
        up_free = r > 0 and art[r - 1][c] != '='
        a = int(rs.choice([0, 1, 2, 3, 4], p=[.7, .08, .08, .1, .04] if up_free
                          else [.05, .4, .4, .1, .05]))
        actions.append(a)
        env.play(a)
      # ... pass 2 replays them through the shared trajectory protocol
      sprites, curtains = [], []
      rec = sprite_recorder('P', sprites)

      def on_frame(env, out):
        rec(env, out)
        curtains.append(env.things['@'].curtain.copy())
      np.random.seed(800 + seed)
      traj = tj.run_trajectory(make, actions, on_frame=on_frame)
    finally:
      ref_shock.LEVELS.pop()
    save('shockwave_%s' % tag, art=tj.art_to_u8(art), actions=np.array(actions, dtype=np.int32),
         sprites=np.array(sprites, dtype=np.int32), curtains=np.stack(curtains).astype(np.uint8),
         numpy_seed=np.array([800 + seed]), **traj)
    print('  shockwave_%s: %d episodes, wins %d, deaths %d' % (
        tag, int(traj['game_over'].sum()), int((traj['reward'] == 1).sum()),
        int((traj['reward'] == -1).sum())))


def groups():
  for seed, margins in ((0, (2, 3)), (1, None), (2, (1, 2))):
    fixture_groups('fixture_groups_%d' % seed, seed, margins)


def better_scrolly(name, level, T=400):
  """better_scrolly_maze stock level + its three croppers (player view with an
  initial offset and no padding, patroller view padded with (None, 3) margins,
  fixed teaser window)."""
  art, offset, teaser = refdriver.ref_better_scrolly_stock(level)
  rs = np.random.RandomState(700 + level)
  actions = rs.randint(0, 5, size=T).tolist()
  sprites, views = [], [[], [], []]
  state = {}

  def make():
    eng = refdriver.ref_better_scrolly(level=level)
    if 'croppers' not in state:
      state['croppers'] = refdriver.ref_better_scrolly_croppers(level)
    for c in state['croppers']:
      c.set_engine(eng)
    return eng

  rec = sprite_recorder('Pabc', sprites)

  def on_frame(env, out):
    rec(env, out)
    for v, c in zip(views, state['croppers']):
      v.append(c.crop(out[0]).board.copy())

  traj = tj.run_trajectory(make, actions, on_frame=on_frame)
  save(name, art=tj.art_to_u8(art), starter_offset=np.array(offset, dtype=np.int32),
       teaser_corner=np.array(teaser, dtype=np.int32),
       actions=np.array(actions, dtype=np.int32), sprites=np.array(sprites, dtype=np.int32),
       view_player=np.stack(views[0]), view_patroller=np.stack(views[1]),
       view_teaser=np.stack(views[2]), **traj)


def fixture_unoccluded(name, seed, T=120):
  """occlusion_in_layers=False (BaseUnoccludedObservationRenderer,
  rendering.py:187-301): per-frame layers of every character."""
  rs = np.random.RandomState(6000 + seed)
  PH, PW, H, W = 13, 17, 7, 10
  pattern = rs.random_sample((PH, PW)) < 0.25
  corner = (int(rs.randint(0, PH - H + 1)), int(rs.randint(0, PW - W + 1)))
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[rs.random_sample((H, W)) < 0.15] = ord('.')
  art[1:4, 2:7] = ord('%')
  art[3, 4] = ord('P')
  art[5, 7] = ord('q')
  art_l = tj.u8_to_art(art)
  walkers = {'P': dict(impassable='#', egocentric=True),
             'q': dict(impassable='', confined=True)}
  scrollys = {'#': dict(pattern=pattern, corner=corner, margins=(2, 3))}
  schedule = [['#'], ['P', 'q', '%']]
  z_order = 'q%#P'
  env = refdriver.ref_fixture(art_l, ' ', walkers, scrollys, drapes='%',
                              update_schedule=schedule, z_order=z_order,
                              occlusion_in_layers=False)
  out = env.its_showtime()
  chars = ''.join(sorted(out[0].layers))
  boards, layers = [], []

  def record(out):
    boards.append(tj.board_of(out[0]).copy())
    layers.append(np.stack([np.array(out[0].layers[c], dtype=bool) for c in chars]))
  record(out)
  motions = rs.randint(0, 9, size=T)
  for m in motions:
    record(env.play(refdriver.fixture_actions_to_ref(int(m))))
  cfg = dict(walkers=walkers,
             scrollys={'#': dict(corner=list(corner), margins=[2, 3])},
             drapes='%', schedule=schedule, z_order=z_order, what_lies_beneath=' ',
             action_chars='', layer_chars=chars)
  save(name, art=art, config=np.frombuffer(json.dumps(cfg).encode(), np.uint8),
       pattern_hash=pattern.astype(np.uint8), actions=motions.astype(np.int32),
       boards=np.stack(boards), layers=np.stack(layers).astype(np.uint8))


def fixture_directives(name, seed, T=250):
  """Walkers + a static drape with Plot directives injected through
  test_things.post_update: rewards, z-order changes, a final termination."""
  tt = refdriver._import()['test_things']
  rs = np.random.RandomState(5000 + seed)
  H, W = 7, 9
  art = np.full((H, W), ord(' '), dtype=np.uint8)
  art[rs.random_sample((H, W)) < 0.2] = ord('#')
  art[2:5, 3:6] = ord('%')                      # static drape region
  for ch, (r, c) in zip('abc', [(1, 1), (5, 7), (3, 4)]):
    art[r, c] = ord(ch)
  art_l = tj.u8_to_art(art)
  walkers = {'a': dict(impassable='#', confined=True),
             'b': dict(impassable='#c', confined=False),
             'c': dict(impassable='', confined=True)}
  schedule = [['a', '%'], ['b', 'c']]
  order = 'a%bc'
  z_order = ''.join(rs.permutation(list(order)))
  engine = refdriver.ref_fixture(art_l, ' ', walkers, drapes='%',
                                 update_schedule=schedule, z_order=z_order)
  out = engine.its_showtime()
  boards = [tj.board_of(out[0]).copy()]
  reward, has_reward, discount, over = [0], [0], [float(out[2])], [0]
  rows, z_orders = [], [list(map(ord, engine.z_order))]
  for t in range(T):
    motions = {ch: int(rs.randint(0, 9)) for ch in 'abc'}
    r = int(rs.randint(-5, 50)) if rs.random_sample() < 0.3 else None
    z = None
    if rs.random_sample() < 0.25:
      this = order[int(rs.randint(4))]
      that = None if rs.random_sample() < 0.3 else order[int(rs.randint(4))]
      if that != this:
        z = (this, that)
    term = (t == T - 1)

    def inject(actions, board, layers, backdrop, things, the_plot, r=r, z=z, term=term):
      if r is not None:
        the_plot.add_reward(r)
      if term:
        the_plot.terminate_episode()
      if z is not None:
        the_plot.change_z_order(*z)
    tt.post_update(engine, 'c', inject)
    out = engine.play(refdriver.fixture_actions_to_ref(motions))
    row = [motions.get(ch, 8) for ch in order]
    row += [-(2 ** 31) if r is None else r, int(term)]
    row += [-1, 0] if z is None else [ord(z[0]), 0 if z[1] is None else ord(z[1])]
    rows.append(row)
    boards.append(tj.board_of(out[0]).copy())
    reward.append(0 if out[1] is None else int(out[1]))
    has_reward.append(0 if out[1] is None else 1)
    discount.append(float(out[2]))
    over.append(int(engine.game_over))
    z_orders.append(list(map(ord, engine.z_order)))
  cfg = dict(walkers=walkers, scrollys={}, drapes='%', schedule=schedule,
             z_order=z_order, what_lies_beneath=' ', action_chars=order)
  save(name, art=art, config=np.frombuffer(json.dumps(cfg).encode(), np.uint8),
       actions=np.array(rows, dtype=np.int64), boards=np.stack(boards),
       reward=np.array(reward, dtype=np.int64),
       has_reward=np.array(has_reward, dtype=np.uint8),
       discount=np.array(discount, dtype=np.float64),
       game_over=np.array(over, dtype=np.uint8),
       z_orders=np.array(z_orders, dtype=np.uint8))


def cropper(name, pad, margins, offset, saccade, T=300):
  cropping = refdriver._import()['cropping']
  maze, board, beneath = levels.scrolly_maze_level(5, world_shape=(65, 65),
                                                   board_shape=(32, 32))
  rs = np.random.RandomState(11)
  actions = rs.randint(0, 5, size=T)
  crops, corners = [], []
  state = {}

  def make():
    eng = refdriver.ref_scrolly_maze(maze, board, beneath)
    if 'c' not in state:
      state['c'] = cropping.ScrollingCropper(
          rows=9, cols=9, to_track=['P'], scroll_margins=margins,
          pad_char=pad, initial_offset=offset, saccade=saccade)
    state['c'].set_engine(eng)
    return eng

  def on_frame(env, out):
    crops.append(state['c'].crop(out[0]).board.copy())
    corners.append(list(state['c']._corner))

  traj = tj.run_trajectory(make, actions.tolist(), on_frame=on_frame)
  cfg = dict(rows=9, cols=9, pad=pad, margins=list(margins),
             offset=None if offset is None else list(offset), saccade=saccade)
  save(name, maze_art=tj.art_to_u8(maze), board_art=tj.art_to_u8(board),
       beneath=np.array([ord(beneath)], dtype=np.uint8),
       config=np.frombuffer(json.dumps(cfg).encode(), np.uint8),
       actions=actions.astype(np.int32), crops=np.stack(crops),
       corners=np.array(corners, dtype=np.int32), **traj)


def classic(name, kind, art, actions):
  """examples/classics game; rewards are Python floats there, so the fixture
  also records the reward's type."""
  sprites, kinds = [], []

  def on_frame(env, out):
    sprite_recorder('P', sprites)(env, out)
    kinds.append(0 if out[1] is None else (2 if isinstance(out[1], float) else 1))
  stock = refdriver.ref_classic_art(kind)
  traj = tj.run_trajectory(lambda: refdriver.ref_classic(kind, art), actions, on_frame=on_frame)
  save(name, art=tj.art_to_u8(art or stock),
       kind=np.frombuffer(kind.encode(), dtype=np.uint8),
       actions=np.array(actions, dtype=np.int32),
       sprites=np.array(sprites, dtype=np.int32),
       reward_type=np.array(kinds, dtype=np.uint8), **traj)


def main():
  assert refdriver.available(), refdriver.MISSING
  if sys.argv[1:] == ['classics']:      # add these without rewriting the older files
    return classics()
  if sys.argv[1:] == ['stories']:
    return stories()
  if sys.argv[1:] == ['fluvial']:
    return fluvials()
  if sys.argv[1:] == ['aperture']:
    return apertures()
  if sys.argv[1:] == ['groups']:
    return groups()
  if sys.argv[1:] == ['ordeal']:
    return ordeals()
  if sys.argv[1:] == ['hello']:
    return hellos()
  if sys.argv[1:] == ['apprehend']:
    return apprehends()
  if sys.argv[1:] == ['shockwave']:
    return shockwaves()
  # BASELINE.json configs[0]: stock scrolly_maze, 1000 random-action steps.
  for level, T in ((0, 1000), (1, 400), (2, 400)):
    maze, board, beneath = refdriver.ref_stock_scrolly_art(level)
    rs = np.random.RandomState(100 + level)
    scrolly('scrolly_stock_L%d' % level, maze, board, beneath,
            rs.randint(0, 5, size=T).tolist(), level=level)
  maze, board, beneath = refdriver.ref_stock_scrolly_art(0)
  scrolly('scrolly_stock_L0_quit', maze, board, beneath,
          np.random.RandomState(7).randint(0, 6, size=300).tolist(), level=0)
  for seed in (0, 1):
    maze, board, beneath = levels.scrolly_maze_level(seed)
    acts = np.random.RandomState(seed).choice(
        [0, 1, 2, 3, 4], size=300, p=[.3, .15, .3, .15, .1]).tolist()
    scrolly('scrolly_gen64_s%d' % seed, maze, board, beneath, acts)

  for level in (0, 1, 2):
    art, wlb = refdriver.ref_stock_warehouse_art(level)
    warehouse('warehouse_stock_L%d' % level, art, wlb,
              np.random.RandomState(200 + level).randint(0, 5, size=600).tolist(),
              level=level)
  art = levels.warehouse_level(3)
  warehouse('warehouse_gen80_s3', art, ' ',
            np.random.RandomState(3).randint(0, 4, size=250).tolist())

  for seed in (0, 1, 2):
    marauders('marauders_stock_s%d' % seed, seed,
              np.random.RandomState(300 + seed).randint(0, 4, size=1000).tolist())

  for seed in range(6):
    fixture_walkers('fixture_walkers_%d' % seed, seed)
  for seed, margins, ego2 in ((0, (2, 3), 0), (1, None, 1), (2, (1, 1), 0),
                              (3, None, 0), (4, (2, 2), 1), (5, (1, 2), 1)):
    fixture_scrolly('fixture_scrolly_%d' % seed, seed, margins, ego2)

  for seed in range(3):
    fixture_directives('fixture_directives_%d' % seed, seed)
  for level in (0, 1, 2):
    better_scrolly('better_stock_L%d' % level, level)
  for seed in range(2):
    fixture_unoccluded('fixture_unoccluded_%d' % seed, seed)

  cropper('crop_ego_pad', ' ', (None, None), None, True)
  cropper('crop_margins_nopad', None, (2, 3), None, True)
  cropper('crop_margins_pad_offset', ' ', (2, 3), (1, -2), False)
  classics()
  stories()
  fluvials()
  apertures()
  groups()
  ordeals()
  hellos()
  apprehends()
  shockwaves()


# Same-shape (4x12) chapters for a list-style story without croppers.
STORY_LIST_CHAPTERS = (
    ('cliff_walk', None),
    ('chain_walk', ['............', '.....P......', '............', '............']),
    ('cliff_walk', ['............', '............', '........P...', '............']),
)


def story_cases():
  """name -> (reference Story builder, actions): see `story()`."""
  st = refdriver.ref_storytelling()
  ref_cropping = refdriver._import()['cropping']

  def classics_list():
    # (A list-story of scrolly_maze levels is not a usable case: the reference
    # copies the old Plot's scrolling-protocol entries into the next game, whose
    # Scrollys then reject the stale order with scrolling.Error.)
    return st.Story([lambda k=k, a=a: refdriver.ref_classic(k, a) for k, a in STORY_LIST_CHAPTERS])

  def classics_cropped():
    def cliff():
      game = refdriver.ref_classic('cliff_walk')
      game.the_plot.next_chapter = 'chain'
      return game

    def rooms():
      game = refdriver.ref_classic('four_rooms')
      game.the_plot.next_chapter = 'cliff'
      return game
    return st.Story(
        {'rooms': rooms, 'cliff': cliff, 'chain': lambda: refdriver.ref_classic('chain_walk')},
        first_chapter='rooms',
        croppers={'rooms': ref_cropping.FixedCropper((1, 0), 4, 12), 'cliff': None,
                  'chain': ref_cropping.FixedCropper((0, 0), 4, 12, pad_char='.')})

  rs = np.random.RandomState(77)
  a1 = rs.randint(0, 5, size=700)
  a1[rs.random_sample(700) < 0.01] = 5              # quit now and then: next chapter
  a2 = rs.randint(0, 4, size=900)
  return {'story_classics_list': (classics_list, (a1 % 4).tolist()),
          'story_classics_cropped': (classics_cropped, a2.tolist())}


def story(name, make, actions):
  """A reference Story played to its end (then rebuilt, like any env of the
  trajectory protocol); also records which chapter was current each frame."""
  chapters = []
  traj = tj.run_trajectory(
      make, actions,
      on_frame=lambda env, out: chapters.append(str(env.the_plot.this_chapter)))
  save(name, actions=np.array(actions, dtype=np.int32),
       chapters=np.array(chapters), **traj)


def stories():
  for name, (make, actions) in story_cases().items():
    story(name, make, actions)


def fluvial(name, art, actions):
  """examples/fluvial_natation.py; also records the (mutable) backdrop curtain."""
  sprites, curtains = [], []

  def on_frame(env, out):
    sprite_recorder('P', sprites)(env, out)
    curtains.append(env.backdrop.curtain.copy())
  traj = tj.run_trajectory(lambda: refdriver.ref_fluvial(art), actions, on_frame=on_frame)
  save(name, art=tj.art_to_u8(art), actions=np.array(actions, dtype=np.int32),
       sprites=np.array(sprites, dtype=np.int32),
       backdrops=np.stack(curtains).astype(np.uint8), **traj)


def aperture(name, level, actions):
  """examples/aperture.py stock level; records the player registers and the
  aperture curtain each frame."""
  sprites, curtains = [], []

  def on_frame(env, out):
    sprite_recorder('A', sprites)(env, out)
    curtains.append(env.things['X'].curtain.copy())
  traj = tj.run_trajectory(lambda: refdriver.ref_aperture(level), actions, on_frame=on_frame)
  save(name, art=tj.art_to_u8(refdriver.ref_aperture_art(level)),
       actions=np.array(actions, dtype=np.int32), sprites=np.array(sprites, dtype=np.int32),
       curtains=np.stack(curtains).astype(np.uint8), **traj)


def apertures():
  for level in (0, 1, 2):
    rs = np.random.RandomState(40 + level)
    actions = rs.choice(list(range(10)), size=900,
                        p=[.14, .14, .14, .14, .04, .1, .1, .1, .095, .005])
    aperture('aperture_stock_L%d' % level, level, actions.tolist())
  aperture('aperture_script_L0', 0, APERTURE_SCRIPT_L0)


# Level 0 played to the cranachan: two aperture pairs, two teleports, reward 1.
APERTURE_SCRIPT_L0 = [8, 7, 1, 1, 2, 1, 1, 1, 1, 1, 6, 8, 3, 3, 1, 1, 1, 3, 4, 0]


def fluvials():
  for which, art in (('stock', refdriver.ref_fluvial_art()), ('other', levels.fluvial_level())):
    actions = np.random.RandomState(len(which)).choice([0, 1, 2], size=800, p=[.2, .6, .2])
    fluvial('fluvial_%s' % which, art, actions.tolist())


def classics():
  for kind in ('four_rooms', 'cliff_walk', 'chain_walk'):
    n_actions = 3 if kind == 'chain_walk' else 6
    for which, art in (('stock', None), ('other', levels.classic_level(kind))):
      actions = np.random.RandomState(len(kind) + len(which)).randint(0, n_actions, size=1200)
      classic('classic_%s_%s' % (kind, which), kind, art, actions.tolist())


if __name__ == '__main__':
  main()
