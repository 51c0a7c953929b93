"""Lower a set-up `Engine` (Python entity objects) to a device game description.

"Recognise and lower" (SURVEY.md §7 H1): game logic upstream is arbitrary Python
in `update()` methods, which cannot run on a GPU.  The fused step kernels
implement the logic of a fixed set of entity classes — the prefabs plus the
concrete classes of the configured example games — and this module maps a
finished `Engine` onto one of those device programs by class identity:

  * an entity class is recognised by (defining module's last name component,
    class name), looked up along its MRO, and only if `update` is not
    overridden below the recognised class;
  * the example modules may be the reference's own files
    (`pycolab/examples/*.py`, imported through `pycolab_b200.compat`) or this
    package's `pycolab_b200/games/*.py`;
  * everything the constructors decided (positions, visibility, curtains,
    patterns, margins, impassable sets, z-order, update groups) is read from
    the live objects, so `make_game()` code runs unchanged.

Anything else raises `NotLoweredError`; there is no CPU fallback.
"""

import numpy as np

from pycolab_b200 import _lib
from pycolab_b200 import things
from pycolab_b200.errors import NotLoweredError
from pycolab_b200.prefab_parts import drapes as prefab_drapes
from pycolab_b200.prefab_parts import sprites as prefab_sprites

# (module tail, class name) -> device role.
LOWERED_CLASSES = {
    ('scrolly_maze', 'PlayerSprite'): 'scrolly.player',
    ('scrolly_maze', 'PatrollerSprite'): 'scrolly.patroller',
    ('scrolly_maze', 'MazeDrape'): 'scrolly.maze',
    ('scrolly_maze', 'CashDrape'): 'scrolly.cash',
    ('warehouse_manager', 'BoxSprite'): 'warehouse.box',
    ('warehouse_manager', 'JudgeDrape'): 'warehouse.judge',
    ('warehouse_manager', 'PlayerSprite'): 'warehouse.player',
    ('extraterrestrial_marauders', 'PlayerSprite'): 'marauders.player',
    ('extraterrestrial_marauders', 'BunkerDrape'): 'marauders.bunker',
    ('extraterrestrial_marauders', 'MarauderDrape'): 'marauders.marauder',
    ('extraterrestrial_marauders', 'UpwardLaserBoltSprite'): 'marauders.up_bolt',
    ('extraterrestrial_marauders', 'DownwardLaserBoltSprite'): 'marauders.down_bolt',
    ('better_scrolly_maze', 'PlayerSprite'): 'better.player',
    ('better_scrolly_maze', 'PatrollerSprite'): 'better.patroller',
    ('better_scrolly_maze', 'CashDrape'): 'better.cash',
    ('four_rooms', 'PlayerSprite'): 'classics.four_rooms',
    ('cliff_walk', 'PlayerSprite'): 'classics.cliff_walk',
    ('chain_walk', 'PlayerSprite'): 'classics.chain_walk',
    ('fluvial_natation', 'PlayerSprite'): 'classics.fluvial',
    ('aperture', 'PlayerSprite'): 'aperture.player',
    ('aperture', 'ApertureDrape'): 'aperture.drape',
    ('hello_world', 'SlidingSprite'): 'hello.slider',
    ('hello_world', 'RollingDrape'): 'hello.roller',
    ('shockwave', 'PlayerSprite'): 'shockwave.player',
    ('shockwave', 'ShockwaveDrape'): 'shockwave.wave',
    ('shockwave', 'MinimalDrape'): 'shockwave.minimal',
    ('apprehend', 'PlayerSprite'): 'apprehend.player',
    ('apprehend', 'BallSprite'): 'apprehend.ball',
    ('ordeal', 'PlayerSprite'): 'ordeal.player',
    ('ordeal', 'DragonduckSprite'): 'ordeal.dragonduck',
    ('ordeal', 'SwordDrape'): 'ordeal.sword',
    ('box_world', 'PlayerSprite'): 'box_world.player',
    ('box_world', 'GemDrape'): 'box_world.gem',
    ('box_world', 'KeyDrape'): 'box_world.key',
    ('box_world', 'LockDrape'): 'box_world.lock',
    # General entities: the reference's test fixtures and this package's twins.
    ('test_things', 'TestMazeWalker'): 'fixture.walker',
    ('test_things', 'TestScrolly'): 'fixture.scrolly',
    ('test_things', 'TestDrape'): 'fixture.drape',
    ('fixtures', 'FixtureMazeWalker'): 'fixture.walker',
    ('fixtures', 'FixtureScrolly'): 'fixture.scrolly',
    ('fixtures', 'FixtureDrape'): 'fixture.drape',
}

# Base classes that hold part of a lowered class's rules without being lowered
# themselves: a class from outside this package that derives from one must carry the
# original's source for it too (BoxThing.is_locked_at / where_player_over_me).
FINGERPRINTED_BASES = {('box_world', 'BoxThing')}

# Backdrop subclasses whose update() has a device counterpart.
LOWERED_BACKDROPS = {
    ('fluvial_natation', 'RiverBackdrop'): 'river',
}

_PROGRAM_OF = {'scrolly': _lib.PROG_SCROLLY_MAZE, 'warehouse': _lib.PROG_WAREHOUSE,
               'marauders': _lib.PROG_MARAUDERS}


def source_fingerprint(text):
  """sha256 over the token stream of `text` (a class definition): comments,
  blank lines and the amount of indentation do not count, everything else does."""
  import hashlib
  import io
  import textwrap
  import tokenize
  skip = (tokenize.COMMENT, tokenize.NL, tokenize.NEWLINE, tokenize.ENCODING,
          tokenize.ENDMARKER)
  h = hashlib.sha256()
  for tok in tokenize.generate_tokens(io.StringIO(textwrap.dedent(text)).readline):
    if tok.type in skip:
      continue
    if tok.type in (tokenize.INDENT, tokenize.DEDENT):
      h.update(b'<%d>' % tok.type)
    else:
      h.update(tok.string.encode('utf-8') + b'\0')
  return h.hexdigest()


def _is_known_implementation(klass, key):
  """Is `klass` one of the implementations the device program was written from?

  Classes of this package (`pycolab_b200.games.*`: set-up twins whose update()
  only says "runs on the device") are trusted by module.  Any other module —
  the reference's own example file loaded through `compat`, or a user's copy of
  it — must match the reference's source for that class token for token: a copy
  with an edited update() (another reward, rule or termination) would otherwise
  be silently replaced by the stock kernel."""
  if klass.__module__.startswith('pycolab_b200.'):
    return True
  from pycolab_b200 import _fingerprints
  want = _fingerprints.KNOWN.get(key)
  if want is None:
    return False
  import inspect
  try:
    text = inspect.getsource(klass)
  except (OSError, TypeError):
    return False
  try:
    return source_fingerprint(text) == want
  except Exception:              # noqa: BLE001 - unparsable source is not a known class
    return False


def role_of(entity):
  """Device role of `entity`, or raise NotLoweredError."""
  cls = type(entity)
  for klass in cls.__mro__:
    key = (klass.__module__.rsplit('.', 1)[-1], klass.__name__)
    if key in LOWERED_CLASSES:
      if cls.update is not klass.update:
        raise NotLoweredError(
            '{} overrides update() of the lowered class {}.{}'.format(
                cls.__name__, *key))
      if not _is_known_implementation(klass, key):
        raise NotLoweredError(
            'class {}.{} is named like the lowered class {}.{} but its source differs '
            'from the implementation the device program restates; edited copies are not '
            'replaced by the stock kernel'.format(klass.__module__, klass.__name__, *key))
      return LOWERED_CLASSES[key]
  raise NotLoweredError(
      'no device program for entity class {}.{} (character {!r}); lowered classes: '
      '{}'.format(cls.__module__, cls.__name__, getattr(entity, 'character', '?'),
                  sorted('%s.%s' % k for k in LOWERED_CLASSES)))


def round_up(x, m):
  return (x + m - 1) // m * m


def pack_rows(mask, words):
  """bool [R, C] -> uint32 [R, words]; cell c is bit c&31 of word c>>5."""
  mask = np.asarray(mask, dtype=bool)
  rows, cols = mask.shape
  assert words * 32 >= cols
  padded = np.zeros((rows, words * 32), dtype=np.uint8)
  padded[:, :cols] = mask
  packed = np.packbits(padded.reshape(rows, words, 32), axis=2, bitorder='little')
  return np.ascontiguousarray(packed).view('<u4').reshape(rows, words)


def unpack_rows(packed, cols):
  packed = np.ascontiguousarray(packed, dtype='<u4')
  rows, words = packed.shape
  bits = np.unpackbits(packed.view(np.uint8).reshape(rows, words * 4), axis=1,
                       bitorder='little')
  return bits[:, :cols].astype(bool)


def char_set_mask(chars):
  out = [0, 0, 0, 0]
  for ch in chars:
    code = ord(ch)
    if code > 127:
      raise NotLoweredError('non-ASCII impassable character {!r}'.format(ch))
    out[code >> 5] |= 1 << (code & 31)
  return out


class LoweredGame(object):
  """One level's device description: spec fields + template arrays."""

  def __init__(self):
    self.program = 0
    self.rows = self.cols = self.pitch = 0
    self.sprite_chars = ''
    self.drape_chars = ''
    self.impassable = []
    self.confined = []
    self.egocentric = []
    self.margins = []
    self.z_order = ''
    self.groups = []
    self.pattern_rows = self.pattern_cols = self.pattern_words = 0
    self.bits_words = 0
    self.backdrop = None        # u8 [H, pitch]
    self.patterns = {}          # drape index -> u32 [PH, PWW]
    self.pattern_mutable = {}   # drape index -> bool
    self.bits = {}              # drape index -> u32 [H, BW]
    self.sprites = None         # i32 [S, 8]
    self.drapes = None          # i32 [D, 8]
    self.plot = None            # i32 [16]
    self.needs_rng = False
    self.rng_kind = 'numpy'     # whose MT19937 stream the device continues: NumPy's legacy
                                # RandomState ('numpy') or Python's `random` ('python')
    self.backdrop_chars = ''
    self.drape_kind = None      # per drape: 1 = Scrolly (fixture program only)
    self.dynamic_z = False      # per-env z-order array (Plot.change_z_order)
    self.program_arg = [0] * 8  # pcl_spec.program_arg
    self.reward_type = int      # the reference's reward type (classics pay floats)
    self.backdrop_role = None   # device counterpart of a Backdrop with update() logic
    self.scroll_groups = ['']   # names of the scrolling groups, index = device group id
    self.sprite_group = []      # per sprite: index into scroll_groups
    self.drape_group = []       # per drape
    self.group_records = None   # i32 [MAX_SCROLL_GROUPS, 4] reset template (groups >= 1)
    self.sync_plot = None       # callable(engine, plot words): mirror device plot state into
                                # the Python Plot after a step (games that keep dict entries)

  def signature(self):
    """Everything that must agree between envs sharing one handle."""
    return (self.program, self.rows, self.cols, self.sprite_chars, self.drape_chars,
            tuple(map(tuple, self.impassable)), tuple(self.confined),
            tuple(self.egocentric), tuple(map(tuple, self.margins)), self.z_order,
            tuple(self.groups), self.pattern_rows, self.pattern_cols,
            tuple(self.program_arg), tuple(self.scroll_groups), tuple(self.sprite_group),
            tuple(self.drape_group))

  def make_spec(self, auto_reset):
    s = _lib.Spec()
    s.abi_version = _lib.ABI_VERSION
    s.program = self.program
    s.rows, s.cols, s.pitch = self.rows, self.cols, self.pitch
    s.n_sprites, s.n_drapes = len(self.sprite_chars), len(self.drape_chars)
    s.auto_reset = 1 if auto_reset else 0
    s.pattern_rows, s.pattern_cols = self.pattern_rows, self.pattern_cols
    s.pattern_words, s.bits_words = self.pattern_words, self.bits_words
    for i, ch in enumerate(self.sprite_chars):
      s.sprite_char[i] = ord(ch)
      for w in range(4):
        s.impassable[i][w] = self.impassable[i][w]
      s.sprite_confined[i] = int(self.confined[i])
      s.sprite_egocentric[i] = int(self.egocentric[i])
    for i, ch in enumerate(self.drape_chars):
      s.drape_char[i] = ord(ch)
      s.margins[i][0], s.margins[i][1] = self.margins[i]
      if self.drape_kind is not None:
        s.drape_kind[i] = self.drape_kind[i]
    for i, ch in enumerate(self.z_order):
      s.z_order[i] = ord(ch)
    for i, v in enumerate(self.program_arg):
      s.program_arg[i] = int(v)
    s.n_scroll_groups = len(self.scroll_groups)
    for i, g in enumerate(self.sprite_group):
      s.sprite_group[i] = g
    for i, g in enumerate(self.drape_group):
      s.drape_group[i] = g
    s.n_groups = len(self.groups)
    k = 0
    for g, group in enumerate(self.groups):
      s.group_len[g] = len(group)
      for ch in group:
        s.group_chars[k] = ord(ch)
        k += 1
    return s


def _sprite_record(sprite, aux0=0, aux1=0, aux2=0):
  if isinstance(sprite, prefab_sprites.MazeWalker):
    vrow, vcol = sprite.virtual_position
    prior = sprite._prior_visible
  else:
    vrow, vcol = sprite.position
    prior = None
  flags = (1 if sprite.visible else 0) | ((0 if prior is None else 2 if prior else 1) << 1)
  return [int(sprite.position[0]), int(sprite.position[1]), int(vrow), int(vcol),
          flags, int(aux0), int(aux1), int(aux2)]


def _walker_meta(sprite, named_groups=False):
  if not isinstance(sprite, prefab_sprites.MazeWalker):
    raise NotLoweredError('sprite {!r} is not a MazeWalker'.format(sprite.character))
  if sprite._scrolling_group != '' and not named_groups:
    raise NotLoweredError('named scrolling groups are lowered by the general program only')
  if (type(sprite)._on_board_exit is not prefab_sprites.MazeWalker._on_board_exit or
      type(sprite)._on_board_enter is not prefab_sprites.MazeWalker._on_board_enter):
    raise NotLoweredError('overridden MazeWalker board exit/enter hooks are not lowered')
  return (char_set_mask(sprite.impassable), bool(sprite._confined_to_board),
          bool(sprite._egocentric_scroller))


def _plot_record(**words):
  rec = [0] * _lib.PLOT_WORDS
  rec[_lib.P_FRAME] = -1
  rec[_lib.P_ORDER_FRAME] = _lib.NEVER
  for name, value in words.items():
    rec[getattr(_lib, 'P_' + name.upper())] = int(value)
  return rec


def _common(engine, game, program):
  game.program = program
  game.rows, game.cols = engine.rows, engine.cols
  game.pitch = round_up(engine.cols, 16)
  game.bits_words = (engine.cols + 31) // 32 + 1
  game.z_order = ''.join(engine.z_order)
  game.groups = [''.join(e.character for e in entities)
                 for _, entities in sorted(engine._update_groups.items())]
  backdrop = engine.backdrop
  game.backdrop_role = None
  if type(backdrop).update is not things.Backdrop.update:
    for klass in type(backdrop).__mro__:
      key = (klass.__module__.rsplit('.', 1)[-1], klass.__name__)
      if (key in LOWERED_BACKDROPS and type(backdrop).update is klass.update and
          _is_known_implementation(klass, key)):
        game.backdrop_role = LOWERED_BACKDROPS[key]
        break
    else:
      raise NotLoweredError('no device program for the update() logic of Backdrop class '
                            '{}.{}'.format(type(backdrop).__module__, type(backdrop).__name__))
  game.backdrop = np.zeros((engine.rows, game.pitch), dtype=np.uint8)
  game.backdrop[:, :engine.cols] = backdrop.curtain
  game.backdrop_chars = ''.join(sorted(backdrop.palette))
  # Unoccluded layers (rendering.py:187-301) change what `layers[...]` look-ups
  # inside update() see; only programs whose logic never reads layers keep
  # their semantics, so only those accept occlusion_in_layers=False.
  if not engine._occlusion_in_layers and program not in (_lib.PROG_SCROLLY_MAZE,
                                                         _lib.PROG_FIXTURE):
    raise NotLoweredError('occlusion_in_layers=False is lowered only for games whose '
                          'entities never consult `layers`')


def _set_sprites(game, sprites, records, named_groups=False):
  game.sprite_chars = ''.join(s.character for s in sprites)
  meta = [_walker_meta(s, named_groups) for s in sprites]
  game.impassable = [m[0] for m in meta]
  game.confined = [m[1] for m in meta]
  game.egocentric = [m[2] for m in meta]
  game.sprites = np.array(records, dtype=np.int32).reshape(len(sprites), _lib.SPRITE_WORDS)


def _scrolly_record(drape, aux0=0, aux1=0):
  r, c = drape._northwest_corner
  return [int(r), int(c), int(r), int(c), _lib.NEVER, int(aux0), int(aux1), 0]


def _lower_scrolly_maze(engine, roles):
  th = engine.things
  want = {'P': 'scrolly.player', 'a': 'scrolly.patroller', 'b': 'scrolly.patroller',
          'c': 'scrolly.patroller', '#': 'scrolly.maze', '@': 'scrolly.cash'}
  if roles != want:
    raise NotLoweredError('scrolly_maze program needs exactly {} (got {})'.format(want, roles))
  game = LoweredGame()
  _common(engine, game, _lib.PROG_SCROLLY_MAZE)
  sprites = [th[c] for c in 'Pabc']
  records = [_sprite_record(th['P'], aux0=0, aux1=_lib.NEVER)]
  records += [_sprite_record(th[c], aux0=int(bool(th[c]._moving_east))) for c in 'abc']
  _set_sprites(game, sprites, records)
  walls, coins = th['#'], th['@']
  for d in (walls, coins):
    if d._scrolling_group != '':
      raise NotLoweredError('only the default scrolling group is lowered')
    if d.whole_pattern.shape != walls.whole_pattern.shape:
      raise NotLoweredError('Scrolly patterns of different shapes')
    if tuple(d._board_shape) != (engine.rows, engine.cols):
      raise NotLoweredError('Scrolly board_shape differs from the Engine board')
  game.drape_chars = '#@'
  game.margins = [(-1, -1) if d._scroll_margins is None else tuple(d._scroll_margins)
                  for d in (walls, coins)]
  game.pattern_rows, game.pattern_cols = walls.whole_pattern.shape
  # zero-padded row: the kernel stages 2 * ceil((63 + W) / 64) words per window row
  # starting at an even word (4 words up to 64 columns).
  slack = 3 if engine.cols <= 64 else 2 * ((63 + engine.cols + 63) // 64) + 1
  game.pattern_words = round_up((game.pattern_cols + 31) // 32 + slack, 2)
  game.patterns = {0: pack_rows(walls.whole_pattern, game.pattern_words),
                   1: pack_rows(coins.whole_pattern, game.pattern_words)}
  game.pattern_mutable = {0: False, 1: True}
  game.drapes = np.array([_scrolly_record(walls), _scrolly_record(coins, -1, -1)],
                         dtype=np.int32)
  game.plot = np.array(_plot_record(aux0=int(coins.whole_pattern.sum())), dtype=np.int32)
  return game


def _lower_warehouse(engine, roles):
  th = engine.things
  groups = [[e.character for e in ents]
            for _, ents in sorted(engine._update_groups.items())]
  if len(groups) != 3 or groups[1] != ['X'] or groups[2] != ['P']:
    raise NotLoweredError('warehouse program needs update groups [boxes, [X], [P]]')
  boxes = groups[0]
  for ch in boxes:
    if roles.get(ch) != 'warehouse.box':
      raise NotLoweredError('unexpected entity {!r} in the box group'.format(ch))
  if roles.get('X') != 'warehouse.judge' or roles.get('P') != 'warehouse.player':
    raise NotLoweredError('warehouse program needs JudgeDrape X and PlayerSprite P')
  game = LoweredGame()
  _common(engine, game, _lib.PROG_WAREHOUSE)
  sprites = [th[c] for c in boxes] + [th['P']]
  _set_sprites(game, sprites, [_sprite_record(s) for s in sprites])
  judge = th['X']
  if judge.curtain.any():
    raise NotLoweredError("a pre-filled 'X' curtain is not lowered")
  game.drape_chars = 'X'
  game.margins = [(-1, -1)]
  rec = [0] * _lib.DRAPE_WORDS
  rec[_lib.D_LAST_FRAME] = _lib.NEVER
  rec[_lib.D_AUX0] = int(judge._last_num_boxes_on_goals)
  game.drapes = np.array([rec], dtype=np.int32)
  game.plot = np.array(_plot_record(), dtype=np.int32)
  if '_' not in engine.backdrop.palette:
    raise NotLoweredError("warehouse backdrop has no goal character '_'")
  return game


def _lower_marauders(engine, roles):
  th = engine.things
  want = {'P': 'marauders.player', 'B': 'marauders.bunker', 'X': 'marauders.marauder',
          'a': 'marauders.up_bolt', 'b': 'marauders.up_bolt', 'c': 'marauders.up_bolt',
          'd': 'marauders.up_bolt', 'y': 'marauders.down_bolt', 'z': 'marauders.down_bolt'}
  if roles != want:
    raise NotLoweredError('marauders program needs exactly {} (got {})'.format(want, roles))
  game = LoweredGame()
  _common(engine, game, _lib.PROG_MARAUDERS)
  sprites = [th[c] for c in 'Pabcdyz']
  _set_sprites(game, sprites, [_sprite_record(s) for s in sprites])
  game.drape_chars = 'BX'
  game.margins = [(-1, -1), (-1, -1)]
  game.bits = {0: pack_rows(th['B'].curtain, game.bits_words),
               1: pack_rows(th['X'].curtain, game.bits_words)}
  recs = []
  for ch in 'BX':
    rec = [0] * _lib.DRAPE_WORDS
    rec[_lib.D_LAST_FRAME] = _lib.NEVER
    recs.append(rec)
  recs[1][_lib.D_AUX0] = int(th['X']._dx)
  game.drapes = np.array(recs, dtype=np.int32)
  game.plot = np.array(_plot_record(aux0=_lib.NEVER, aux1=_lib.NEVER), dtype=np.int32)
  game.needs_rng = True
  return game


def _lower_better_scrolly(engine, roles):
  th = engine.things
  want = {'P': 'better.player', 'a': 'better.patroller', 'b': 'better.patroller',
          'c': 'better.patroller', '@': 'better.cash'}
  if roles != want:
    raise NotLoweredError('better_scrolly_maze program needs exactly {} (got {})'.format(
        want, roles))
  game = LoweredGame()
  _common(engine, game, _lib.PROG_BETTER_SCROLLY)
  sprites = [th[c] for c in 'Pabc']
  records = [_sprite_record(th['P'])]
  records += [_sprite_record(th[c], aux0=int(bool(th[c]._moving_east))) for c in 'abc']
  _set_sprites(game, sprites, records)
  game.drape_chars = '@'
  game.margins = [(-1, -1)]
  game.bits = {0: pack_rows(th['@'].curtain, game.bits_words)}
  rec = [0] * _lib.DRAPE_WORDS
  rec[_lib.D_LAST_FRAME] = _lib.NEVER
  game.drapes = np.array([rec], dtype=np.int32)
  game.plot = np.array(_plot_record(aux0=int(th['@'].curtain.sum())), dtype=np.int32)
  return game


def _lower_classics(engine, roles):
  """examples/classics: one MazeWalker 'P', no drapes; the rule set rides in
  pcl_spec.program_arg (four_rooms.py:78 fixes the goal cell at (4, 3))."""
  if list(roles) != ['P']:
    raise NotLoweredError('classics programs have exactly one entity, P (got {})'.format(roles))
  game = LoweredGame()
  _common(engine, game, _lib.PROG_CLASSICS)
  rule = roles['P'].split('.')[1]
  game.program_arg[0] = {'four_rooms': _lib.CLASSIC_FOUR_ROOMS,
                         'cliff_walk': _lib.CLASSIC_CLIFF_WALK,
                         'chain_walk': _lib.CLASSIC_CHAIN_WALK,
                         'fluvial': _lib.CLASSIC_FLUVIAL}[rule]
  if rule == 'four_rooms':
    game.program_arg[1], game.program_arg[2] = 4, 3
  if (rule == 'fluvial') != (game.backdrop_role == 'river'):
    raise NotLoweredError('the river Backdrop and the swimmer are lowered only together')
  if rule == 'fluvial':
    game.program_arg[1], game.program_arg[2] = 1, 4      # curtain[1:4, :], fluvial_natation.py:110
  if game.rows * game.pitch > 8192:
    raise NotLoweredError('classics boards are staged whole in shared memory (<= 8 KiB)')
  player = engine.things['P']
  _set_sprites(game, [player], [_sprite_record(player)])
  if rule == 'fluvial' and any(game.impassable[0]):
    raise NotLoweredError('the river program needs a swimmer with no impassable characters')
  game.drapes = np.zeros((0, _lib.DRAPE_WORDS), dtype=np.int32)
  game.plot = np.array(_plot_record(), dtype=np.int32)
  game.reward_type = int if rule == 'fluvial' else float
  return game


def _lower_hello(engine, roles):
  """examples/hello_world.py:58-118: up to four SlidingSprites (plain Sprites, each
  with one of four diagonal direction sets) and one RollingDrape, one update group."""
  th = engine.things
  sliders = [c for c in ''.join(_update_order(engine)) if roles[c] == 'hello.slider']
  rollers = [c for c, r in roles.items() if r == 'hello.roller']
  if not 1 <= len(sliders) <= 4 or len(rollers) != 1:
    raise NotLoweredError('hello_world program needs 1-4 SlidingSprites and one RollingDrape')
  game = LoweredGame()
  _common(engine, game, _lib.PROG_HELLO)
  if len(game.groups) != 1:
    raise NotLoweredError('hello_world entities share one update group')
  records = []
  for ch in sliders:
    sp = th[ch]
    sets = list(zip(type(sp)._DX, type(sp)._DY))
    try:
      k = sets.index((sp._dx, sp._dy))
    except ValueError:
      raise NotLoweredError('SlidingSprite {!r} uses an unknown direction set'.format(ch))
    records.append(_sprite_record(sp, aux0=k))
  game.sprite_chars = ''.join(sliders)
  game.impassable = [[0, 0, 0, 0]] * len(sliders)
  game.confined = [False] * len(sliders)
  game.egocentric = [False] * len(sliders)
  game.sprites = np.array(records, dtype=np.int32).reshape(len(sliders), _lib.SPRITE_WORDS)
  game.drape_chars = rollers[0]
  game.margins = [(-1, -1)]
  rec = [0] * _lib.DRAPE_WORDS
  rec[_lib.D_LAST_FRAME] = _lib.NEVER
  game.drapes = np.array([rec], dtype=np.int32)
  game.bits[0] = pack_rows(th[rollers[0]].curtain, game.bits_words)   # the un-rolled curtain
  game.plot = np.array(_plot_record(), dtype=np.int32)
  for k, ch in enumerate(game.z_order):          # the kernel paints in this order
    game.program_arg[k] = ord(ch)
  return game


def _f64_words(x):
  """float64 -> (lo, hi) int32 words, as the kernels' __hiloint2double reads them."""
  lo, hi = np.array([x], dtype='<f8').view('<i4')
  return int(lo), int(hi)


def _lower_apprehend(engine, roles):
  """examples/apprehend.py:56-131: the catcher 'P' and the falling ball, one group
  [ball, catcher].  The ball's float64 slope (drawn when the Python sprite was built)
  and accumulator travel as bit patterns; `needs_rng` lets a BATCHED engine draw a new
  slope per episode on the device from per-env `random.Random` states."""
  th = engine.things
  players = [c for c, r in roles.items() if r == 'apprehend.player']
  balls = [c for c, r in roles.items() if r == 'apprehend.ball']
  if len(players) != 1 or len(balls) != 1 or len(roles) != 2:
    raise NotLoweredError('apprehend program needs one PlayerSprite and one BallSprite')
  game = LoweredGame()
  _common(engine, game, _lib.PROG_APPREHEND)
  pl, ball = th[players[0]], th[balls[0]]
  if _update_order(engine) != [balls[0], players[0]] or len(game.groups) != 1:
    raise NotLoweredError('apprehend program needs update_schedule [ball, player]')
  if game.z_order != balls[0] + players[0]:
    raise NotLoweredError('apprehend program draws the player over the ball')
  lo, hi = _f64_words(ball._dx)
  _set_sprites(game, [pl, ball], [_sprite_record(pl), _sprite_record(ball, aux0=lo, aux1=hi)])
  alo, ahi = _f64_words(ball._x_accumulator)
  game.drape_chars = ''
  game.margins = []
  game.drapes = np.zeros((0, _lib.DRAPE_WORDS), dtype=np.int32)
  game.plot = np.array(_plot_record(aux0=alo, aux1=ahi), dtype=np.int32)
  game.needs_rng = True
  game.rng_kind = 'python'
  return game


def _lower_shockwave(engine, roles):
  """examples/shockwave.py:91-197: the player, the ShockwaveDrape and the two static
  MinimalDrapes the wave's update() names by character (' ' danger zone, '^' safe
  zone; walls are the backdrop's '=')."""
  th = engine.things
  by_role = {}
  for ch, role in roles.items():
    by_role.setdefault(role, []).append(ch)
  if (sorted(by_role) != ['shockwave.minimal', 'shockwave.player', 'shockwave.wave'] or
      len(by_role['shockwave.player']) != 1 or len(by_role['shockwave.wave']) != 1 or
      sorted(by_role['shockwave.minimal']) != [' ', '^']):
    raise NotLoweredError("shockwave program needs one PlayerSprite, one ShockwaveDrape and "
                          "MinimalDrapes ' ' and '^' (got {})".format(roles))
  p_ch, w_ch = by_role['shockwave.player'][0], by_role['shockwave.wave'][0]
  game = LoweredGame()
  _common(engine, game, _lib.PROG_SHOCKWAVE)
  order = _update_order(engine)
  if len(game.groups) != 1 or sorted(order[:2]) != [' ', '^'] or order[2:] != [p_ch, w_ch]:
    raise NotLoweredError("shockwave program needs update_schedule [' ', '^', P, wave]")
  if game.z_order != ' ^' + w_ch + p_ch:
    raise NotLoweredError("shockwave program needs z_order [' ', '^', wave, P]")
  pl, wave = th[p_ch], th[w_ch]
  if set(pl.impassable) != {'='}:
    raise NotLoweredError("the wave's update() stops at '=': the player must do the same")
  if engine.rows > 32 or engine.cols > 64:
    raise NotLoweredError('shockwave program: boards up to 32 x 64')
  _set_sprites(game, [pl], [_sprite_record(pl)])
  game.drape_chars = w_ch + ' ^'
  game.margins = [(-1, -1)] * 3
  recs = []
  for _ in range(3):
    rec = [0] * _lib.DRAPE_WORDS
    rec[_lib.D_LAST_FRAME] = _lib.NEVER
    recs.append(rec)
  recs[0][_lib.D_AUX1] = int(wave._steps_since_impact)
  if wave.curtain.any() or np.any(wave._distance_from_impact):
    raise NotLoweredError('a ShockwaveDrape that is already burning is not lowered')
  game.drapes = np.array(recs, dtype=np.int32)
  for d, ch in enumerate(game.drape_chars):
    game.bits[d] = pack_rows(th[ch].curtain, game.bits_words)
  game.plot = np.array(_plot_record(), dtype=np.int32)
  game.program_arg[0] = int(wave._width)
  game.needs_rng = True                         # np.random.randint, shockwave.py:133
  return game


# What the box-world program restates of box_world.py's module constants: an edited
# copy could change them without touching a class body.
_BOX_WORLD_CONSTANTS = {
    'GEM': '*', 'PLAYER': '.', 'BORDER': '#',
    'KEYS': list('abcdefghijklmnopqrst'), 'LOCKS': list('ABCDEFGHIJKLMNOPQRST'),
    'REWARD_GOAL': 10., 'REWARD_STEP': 0., 'REWARD_OPEN_CORRECT': 1.,
    'REWARD_OPEN_WRONG': -1.,
    'ACTION_MAP': {0: (-1, 0), 1: (1, 0), 2: (0, -1), 3: (0, 1)},
}


def _same_constant(got, want):
  if isinstance(want, dict):
    return (isinstance(got, dict) and set(got) == set(want) and
            all(tuple(got[k]) == want[k] for k in want))
  if isinstance(want, float):
    return isinstance(got, (int, float)) and not isinstance(got, bool) and got == want
  return type(got) is type(want) and got == want


def _check_box_world_module(klass):
  """The module that defines `klass` (whose methods read its globals) must hold the
  original's constants."""
  import sys
  module = sys.modules.get(klass.__module__)
  for name, want in _BOX_WORLD_CONSTANTS.items():
    if not _same_constant(getattr(module, name, None), want):
      raise NotLoweredError('box_world program: {}.{} = {!r} differs from the original\'s '
                            '{!r}'.format(klass.__module__, name,
                                          getattr(module, name, None), want))


def _box_world_classes(entity):
  """Classes along the MRO of a box-world entity whose code the device restates: the
  lowered class and, for drapes, BoxThing.  Classes from outside this package must
  carry the original's source; subclasses may not override the rules' helpers."""
  cls = type(entity)
  out = []
  for klass in cls.__mro__:
    key = (klass.__module__.rsplit('.', 1)[-1], klass.__name__)
    if key in LOWERED_CLASSES or key in FINGERPRINTED_BASES:
      if key in FINGERPRINTED_BASES and not _is_known_implementation(klass, key):
        raise NotLoweredError(
            'class {}.{} is named like {}.{} but its source differs from the original\'s; '
            'edited copies are not replaced by the stock kernel'.format(
                klass.__module__, klass.__name__, *key))
      out.append(klass)
  for klass in out:
    for name in ('_in_direction', 'is_locked_at', 'where_player_over_me'):
      if hasattr(klass, name) and getattr(cls, name) is not getattr(klass, name):
        raise NotLoweredError('{} overrides {}() of {}.{}'.format(
            cls.__name__, name, klass.__module__, klass.__name__))
  if (not isinstance(entity, prefab_sprites.MazeWalker) and
      not any(k.__name__ == 'BoxThing' for k in out)):
    raise NotLoweredError('box_world drape {!r} does not derive from BoxThing'.format(
        entity.character))
  return out


def _lower_box_world(engine, roles):
  """examples/research/box_world/box_world.py:127-445: the player '.' and any number
  of key, lock and gem drapes, all in ONE update group [player] + sorted(drapes) and
  drawn in sorted(drapes) + [player].  The drapes never overlap, so they travel as one
  byte plane (pcl.h PCL_PROG_BOX_WORLD): the spec names the player alone, and every
  level of any drape set shares one signature."""
  th = engine.things
  kinds = {'box_world.player': '.', 'box_world.gem': '*'}
  for ch, role in roles.items():
    if role in ('box_world.key', 'box_world.lock'):
      upper = role == 'box_world.lock'
      ok = len(ch) == 1 and ch.isascii() and ch.isalpha() and ch.isupper() == upper and \
          ord(ch.lower()) - ord('a') < 20
    else:
      ok = ch == kinds[role]
    if not ok:
      raise NotLoweredError('box_world program: character {!r} cannot be a {}'.format(
          ch, role.split('.')[1]))
  if list(roles.values()).count('box_world.player') != 1:
    raise NotLoweredError('box_world program needs exactly one PlayerSprite')
  for ent in th.values():
    for klass in _box_world_classes(ent):
      _check_box_world_module(klass)
  game = LoweredGame()
  _common(engine, game, _lib.PROG_BOX_WORLD)
  drapes = sorted(ch for ch in roles if ch != '.')
  if game.groups != ['.' + ''.join(drapes)]:
    raise NotLoweredError('box_world program needs one update group [player] + '
                          'sorted(drapes) (got {})'.format(game.groups))
  if game.z_order != ''.join(drapes) + '.':
    raise NotLoweredError('box_world program needs z_order sorted(drapes) + [player] '
                          '(got {!r})'.format(game.z_order))
  if engine.rows > 32 or engine.cols > 32:
    raise NotLoweredError('box_world program: boards up to 32 x 32 (grid_size <= 30)')
  room = np.full((engine.rows, engine.cols), ord(' '), dtype=np.uint8)
  room[[0, -1], :] = room[:, [0, -1]] = ord('#')
  if not np.array_equal(engine.backdrop.curtain, room):
    raise NotLoweredError("box_world program: the backdrop must be a room of ' ' walled "
                          "by '#'")
  pl = th['.']
  impassable, confined, egocentric = _walker_meta(pl)
  if impassable != char_set_mask('#') or not confined or egocentric:
    raise NotLoweredError("box_world program: the player is confined and stopped by '#' "
                          "alone")
  if not pl.visible or tuple(pl.virtual_position) != tuple(pl.position):
    raise NotLoweredError('box_world program: the player starts visible on the board')
  game.pitch = round_up(engine.cols, 16)
  game.bits_words = game.pitch // 4
  plane = np.zeros((engine.rows, game.pitch), dtype=np.uint8)
  for ch in drapes:
    curtain = th[ch].curtain
    if np.any(plane[:, :engine.cols][curtain]):
      raise NotLoweredError('box_world program: drapes overlap at set-up')
    plane[:, :engine.cols][curtain] = ord(ch)
    if ch in 'ABCDEFGHIJKLMNOPQRST' and th[ch].key_that_opens != ch.lower():
      raise NotLoweredError('box_world lock {!r} opens with {!r}'.format(
          ch, th[ch].key_that_opens))
  if np.any(plane[[0, -1], :]) or np.any(plane[:, [0, engine.cols - 1]]):
    raise NotLoweredError('box_world program: no drape on the wall at set-up')
  for x, y in pl.distractors:
    x, y = int(x), int(y)
    if 0 <= y < engine.rows and 0 <= x < engine.cols and chr(plane[y, x]).isupper():
      plane[y, x] |= 0x80               # only a lock cell's membership is ever asked
  steps, limit = pl._step_counter, pl._max_num_steps
  if not all(isinstance(v, (int, np.integer)) for v in (steps, limit)):
    raise NotLoweredError('box_world program: integer step counts only')
  game.sprite_chars = '.'
  game.impassable = [char_set_mask('#')]
  game.confined = [True]
  game.egocentric = [False]
  game.sprites = np.array([_sprite_record(pl, aux0=steps, aux1=limit)], dtype=np.int32)
  game.z_order = '.'
  game.groups = ['.']
  game.drape_chars = ''
  game.margins = []
  game.drapes = np.zeros((0, _lib.DRAPE_WORDS), dtype=np.int32)
  game.bits = {0: plane}
  game.plot = np.array(_plot_record(), dtype=np.int32)
  game.reward_type = float                      # box_world.py pays 0.0 / 1.0 / -1.0 / 10.0
  return game


def _update_order(engine):
  return [e.character for _, ents in sorted(engine._update_groups.items()) for e in ents]


_ORDEAL_CHAPTERS = {'castle': _lib.ORDEAL_CASTLE, 'cavern': _lib.ORDEAL_CAVERN,
                    'kansas': _lib.ORDEAL_KANSAS}


def _lower_ordeal(engine, roles):
  """examples/ordeal.py:74-266: one chapter of the Story.  Which chapter this Engine
  is comes from its entities (castle: P + D, cavern: P + S, kansas: P) and must agree
  with `the_plot.this_chapter`, which Story set before its_showtime()
  (storytelling.py:453-454).  The Plot entries the game code keeps in dict slots —
  `has_sword`, `last_position` — and the chapter bookkeeping enter the device plot
  record here and are mirrored back after every step (`sync_plot`)."""
  th, plot = engine.things, engine.the_plot
  by_role = sorted(roles.values())
  chapter = {('ordeal.dragonduck', 'ordeal.player'): 'castle',
             ('ordeal.player', 'ordeal.sword'): 'cavern',
             ('ordeal.player',): 'kansas'}.get(tuple(by_role))
  if chapter is None:
    raise NotLoweredError('ordeal program: unknown chapter with entities {}'.format(roles))
  if plot.this_chapter is not None and plot.this_chapter != chapter:
    raise NotLoweredError('ordeal chapter {!r} is running under the Story key {!r}'.format(
        chapter, plot.this_chapter))
  if plot.prior_chapter is not None and plot.prior_chapter not in _ORDEAL_CHAPTERS:
    raise NotLoweredError('ordeal chapter entered from an unknown chapter {!r}'.format(
        plot.prior_chapter))
  game = LoweredGame()
  _common(engine, game, _lib.PROG_ORDEAL)
  if len(game.groups) != 1:
    raise NotLoweredError('ordeal chapters have one update group')
  player = [c for c, r in roles.items() if r == 'ordeal.player'][0]
  sprites = [th[player]] + [th[c] for c, r in roles.items() if r == 'ordeal.dragonduck']
  if game.groups[0][0] != player:
    raise NotLoweredError('the ordeal player must update first')
  if game.rows * game.pitch > 8192:
    raise NotLoweredError('ordeal boards are staged whole in shared memory (<= 8 KiB)')
  _set_sprites(game, sprites, [_sprite_record(s) for s in sprites])
  game.program_arg[0] = _ORDEAL_CHAPTERS[chapter]
  drapes = [c for c, r in roles.items() if r == 'ordeal.sword']
  game.drape_chars = ''.join(drapes)
  game.margins = [(-1, -1)] * len(drapes)
  game.drapes = np.zeros((len(drapes), _lib.DRAPE_WORDS), dtype=np.int32)
  for d, ch in enumerate(drapes):
    game.drapes[d, _lib.D_LAST_FRAME] = _lib.NEVER
    game.bits[d] = pack_rows(th[ch].curtain, game.bits_words)
  last = plot.get('last_position')
  game.plot = np.array(_plot_record(
      aux0=1 if plot.get('has_sword') else 0,
      aux1=-1 if last is None else (int(last[0]) << 16) | int(last[1]),
      aux2=_lib.ORDEAL_NEXT_UNSET,
      aux3=_ORDEAL_CHAPTERS.get(plot.prior_chapter, 0)), dtype=np.int32)
  game.dynamic_z = len(sprites) + len(drapes) == 2      # the kernel reads (castle: rewrites) it
  game.reward_type = float                              # ordeal.py pays 1.0 / -1.0
  names = {v: k for k, v in _ORDEAL_CHAPTERS.items()}

  def sync_plot(eng, words):
    p = eng.the_plot
    if words[_lib.P_AUX0]:
      p['has_sword'] = True
    if words[_lib.P_AUX1] >= 0:
      p['last_position'] = things.Sprite.Position(int(words[_lib.P_AUX1]) >> 16,
                                                  int(words[_lib.P_AUX1]) & 0xffff)
    if words[_lib.P_AUX2] != _lib.ORDEAL_NEXT_UNSET:
      p.next_chapter = names.get(int(words[_lib.P_AUX2]))   # 0 -> None: the story ends
  game.sync_plot = sync_plot
  return game


def _lower_aperture(engine, roles):
  """examples/aperture.py:188-196: sprite 'A' + the aperture drape.  The drape's
  state is its `_apertures` list (at most two cells) in the record's AUX words."""
  players = [c for c, r in roles.items() if r == 'aperture.player']
  drapes = [c for c, r in roles.items() if r == 'aperture.drape']
  if len(players) != 1 or len(drapes) != 1 or len(roles) != 2:
    raise NotLoweredError('aperture program needs one player and one aperture drape '
                          '(got {})'.format(roles))
  game = LoweredGame()
  _common(engine, game, _lib.PROG_APERTURE)
  player, drape = engine.things[players[0]], engine.things[drapes[0]]
  if game.z_order != drapes[0] + players[0] or game.groups != [players[0], drapes[0]]:
    raise NotLoweredError('aperture program needs update groups [[player], [drape]] and the '
                          'player drawn over the drape')
  if drape.curtain.any() or list(drape._apertures) != [None, None]:
    raise NotLoweredError('the aperture drape must start with no apertures')
  if game.rows * game.pitch > 8192:
    raise NotLoweredError('aperture boards are staged whole in shared memory (<= 8 KiB)')
  _set_sprites(game, [player], [_sprite_record(player)])
  game.drape_chars = drapes[0]
  game.margins = [(-1, -1)]
  rec = [0] * _lib.DRAPE_WORDS
  rec[_lib.D_LAST_FRAME] = _lib.NEVER
  rec[_lib.D_AUX0] = rec[_lib.D_AUX1] = -1
  game.drapes = np.array([rec], dtype=np.int32)
  game.plot = np.array(_plot_record(), dtype=np.int32)
  return game


def _lower_fixture(engine, roles):
  th = engine.things
  game = LoweredGame()
  _common(engine, game, _lib.PROG_FIXTURE)
  order = ''.join(game.groups)
  sprite_chars = [c for c in order if roles[c] == 'fixture.walker']
  drape_chars = [c for c in order if roles[c] != 'fixture.walker']
  if len(sprite_chars) > _lib.MAX_SPRITES or len(drape_chars) > _lib.MAX_DRAPES:
    raise NotLoweredError('too many entities for the general device program')
  sprites = [th[c] for c in sprite_chars]
  _set_sprites(game, sprites, [_sprite_record(s, aux0=0, aux1=_lib.NEVER) for s in sprites],
               named_groups=True)
  # Scrolling groups (protocols/scrolling.py:198-241): one device record per name.
  names = []
  for ch in order:
    name = getattr(th[ch], '_scrolling_group', None)
    if name is not None and name not in names:
      names.append(name)
  names = names or ['']
  if len(names) > _lib.MAX_SCROLL_GROUPS:
    raise NotLoweredError('more than {} scrolling groups'.format(_lib.MAX_SCROLL_GROUPS))
  game.scroll_groups = names
  game.sprite_group = [names.index(th[c]._scrolling_group) for c in sprite_chars]
  game.drape_group = [names.index(getattr(th[c], '_scrolling_group', names[0]))
                      for c in drape_chars]
  game.group_records = np.zeros((_lib.MAX_SCROLL_GROUPS, _lib.GROUP_WORDS), dtype=np.int32)
  game.group_records[:, _lib.G_ORDER_FRAME] = _lib.NEVER
  game.drape_chars = ''.join(drape_chars)
  game.drape_kind, game.margins, recs = [], [], []
  shape = None
  for d, ch in enumerate(drape_chars):
    ent = th[ch]
    if roles[ch] == 'fixture.scrolly':
      if shape not in (None, ent.whole_pattern.shape):
        raise NotLoweredError('Scrolly patterns of different shapes')
      shape = ent.whole_pattern.shape
      game.drape_kind.append(1)
      game.margins.append((-1, -1) if ent._scroll_margins is None
                          else tuple(ent._scroll_margins))
      recs.append(_scrolly_record(ent))
    else:
      game.drape_kind.append(0)
      game.margins.append((-1, -1))
      rec = [0] * _lib.DRAPE_WORDS
      rec[_lib.D_LAST_FRAME] = _lib.NEVER
      recs.append(rec)
      game.bits[d] = pack_rows(ent.curtain, game.bits_words)
  if shape is not None:
    game.pattern_rows, game.pattern_cols = shape
    game.pattern_words = round_up((shape[1] + 31) // 32 + 3, 2)
    for d, ch in enumerate(drape_chars):
      if game.drape_kind[d]:
        game.patterns[d] = pack_rows(th[ch].whole_pattern, game.pattern_words)
        game.pattern_mutable[d] = False
  game.drapes = np.array(recs, dtype=np.int32).reshape(len(drape_chars), _lib.DRAPE_WORDS)
  game.plot = np.array(_plot_record(), dtype=np.int32)
  game.dynamic_z = True
  return game


def lower(engine):
  """`Engine` (set-up finished, not yet showtime) -> `LoweredGame`."""
  roles = {ch: role_of(ent) for ch, ent in engine.things.items()}
  families = {role.split('.')[0] for role in roles.values()}
  if len(families) != 1:
    raise NotLoweredError('entities from different game programs: {}'.format(roles))
  family = families.pop()
  lowerers = {'scrolly': _lower_scrolly_maze, 'warehouse': _lower_warehouse,
              'marauders': _lower_marauders, 'fixture': _lower_fixture,
              'classics': _lower_classics, 'better': _lower_better_scrolly,
              'aperture': _lower_aperture, 'ordeal': _lower_ordeal,
              'hello': _lower_hello, 'apprehend': _lower_apprehend,
              'shockwave': _lower_shockwave, 'box_world': _lower_box_world}
  if family not in lowerers:
    raise NotLoweredError(family)
  game = lowerers[family](engine, roles)
  if game.backdrop_role is not None and family != 'classics':
    raise NotLoweredError('a Backdrop with update() logic is lowered only with its own game')
  return game
