"""`Engine`: the pycolab game engine surface over the B200 step engine.

Set-up API identical to the reference (`pycolab/engine.py:248-518`): the same
methods, argument meaning and exceptions, building the same registry of entity
objects.  `its_showtime()` lowers the finished game to a device program
(`lowering.lower`) and from then on `play()` is one fused CUDA kernel per step
through the C ABI (`BatchedEngine`, batch 1) — the Python `update()` methods
are never executed.  For thousands of envs use `batched.BatchedEngine`
directly; this class is the drop-in single-env view of the same machinery.
"""

import collections

import numpy as np

from pycolab_b200 import _lib
from pycolab_b200 import plot
from pycolab_b200 import rendering
from pycolab_b200 import things
from pycolab_b200.prefab_parts import drapes as prefab_drapes
from pycolab_b200.prefab_parts import sprites as prefab_sprites


class Engine(object):

  def __init__(self, rows, cols, occlusion_in_layers=True):
    self._rows, self._cols = rows, cols
    self._occlusion_in_layers = occlusion_in_layers
    self._the_plot = plot.Plot()
    self._showtime = False
    self._game_over = False
    self._backdrop = None
    self._sprites_and_drapes = collections.OrderedDict()
    self._update_groups = collections.defaultdict(list)
    self._current_update_group = ''
    self._board = None
    self._batched = None
    self._backdrop_template = None   # initial curtain of a Backdrop the device animates

  # ------------------------------------------------------------ set-up API
  def set_backdrop(self, characters, backdrop_class, *args, **kwargs):
    self._no_showtime('set_backdrop')
    return self.set_prefilled_backdrop(
        characters, np.zeros((self._rows, self._cols), dtype=np.uint8),
        backdrop_class, *args, **kwargs)

  def set_prefilled_backdrop(self, characters, prefill, backdrop_class, *args, **kwargs):
    self._no_showtime('set_prefilled_backdrop')
    self._check_chars(characters)
    self._check_unclaimed(characters)
    if self._backdrop:
      raise RuntimeError('A backdrop of type {} has already been supplied to this '
                         'Engine.'.format(type(self._backdrop)))
    if not issubclass(backdrop_class, things.Backdrop):
      raise TypeError('backdrop_class arguments to Engine.set_backdrop must either be a '
                      'Backdrop class or one of its subclasses.')
    curtain = np.zeros((self._rows, self._cols), dtype=np.uint8)
    np.copyto(dst=curtain, src=prefill, casting='equiv')
    self._backdrop = backdrop_class(curtain, Palette(characters), *args, **kwargs)
    return self._backdrop

  def add_drape(self, character, drape_class, *args, **kwargs):
    self._no_showtime('add_drape')
    return self.add_prefilled_drape(
        character, np.zeros((self._rows, self._cols), dtype=np.bool_),
        drape_class, *args, **kwargs)

  def add_prefilled_drape(self, character, prefill, drape_class, *args, **kwargs):
    self._no_showtime('add_prefilled_drape')
    self._check_chars(character, mandatory_len=1)
    self._check_unclaimed(character)
    if not issubclass(drape_class, things.Drape):
      raise TypeError('drape_class arguments to Engine.add_drape must be a subclass of '
                      'Drape')
    curtain = np.zeros((self._rows, self._cols), dtype=np.bool_)
    np.copyto(dst=curtain, src=prefill, casting='equiv')
    drape = drape_class(curtain, character, *args, **kwargs)
    self._sprites_and_drapes[character] = drape
    self._update_groups[self._current_update_group].append(drape)
    return drape

  def add_sprite(self, character, position, sprite_class, *args, **kwargs):
    self._no_showtime('add_sprite')
    self._check_chars(character, mandatory_len=1)
    self._check_unclaimed(character)
    if not issubclass(sprite_class, things.Sprite):
      raise TypeError('sprite_class arguments to Engine.add_sprite must be a subclass of '
                      'Sprite')
    if not (0 <= position[0] < self._rows and 0 <= position[1] < self._cols):
      raise ValueError('Position {} does not fall inside a {}x{} game board.'.format(
          position, self._rows, self._cols))
    corner = things.Sprite.Position(self._rows, self._cols)
    sprite = sprite_class(corner, things.Sprite.Position(*position), character,
                          *args, **kwargs)
    self._sprites_and_drapes[character] = sprite
    self._update_groups[self._current_update_group].append(sprite)
    return sprite

  def update_group(self, group_name):
    self._no_showtime('update_group')
    self._current_update_group = group_name

  def set_z_order(self, z_order):
    self._no_showtime('set_z_order')
    if (set(z_order) != set(self._sprites_and_drapes) or
        len(z_order) != len(self._sprites_and_drapes)):
      raise ValueError('The z_order argument {!r} to Engine.set_z_order is not a proper '
                       'permutation of the characters corresponding to Sprites and '
                       'Drapes in this game, which are {}.'.format(
                           z_order, self._sprites_and_drapes.keys()))
    self._sprites_and_drapes = collections.OrderedDict(
        (ch, self._sprites_and_drapes[ch]) for ch in z_order)

  # -------------------------------------------------------------- running
  def its_showtime(self):
    """engine.py:520-581: freeze the set-up, lower to the device, run frame 0."""
    self._no_showtime('its_showtime')
    if self._backdrop is None:
      raise RuntimeError('its_showtime() called before a Backdrop was supplied')
    from pycolab_b200 import batched
    from pycolab_b200 import lowering
    lowered = lowering.lower(self)          # NotLoweredError if not accelerable
    # Upstream folds directives issued BEFORE its_showtime() into frame 0
    # (engine.py:761-847 runs on whatever the Plot holds).  The device's frame 0 starts
    # from clean directives, so such a set-up is refused rather than silently dropped.
    pending = self._the_plot._engine_directives
    if (pending.z_updates or pending.summed_reward is not None or pending.game_over or
        pending.discount != 1.0):
      from pycolab_b200.errors import NotLoweredError
      raise NotLoweredError('Plot directives issued before its_showtime() (add_reward, '
                            'terminate_episode, change_default_discount, change_z_order) are '
                            'not carried into the device\'s first frame')
    rng_states = None
    if lowered.needs_rng and lowered.rng_kind == 'python':
      # apprehend.py:103 draws in the sprite's constructor, which has already run
      # (from the global `random`, as upstream): the device takes the drawn value
      # from the template and needs no generator for this one episode.
      rng_states = False
    elif lowered.needs_rng:
      # Upstream game code draws from the GLOBAL NumPy RNG
      # (extraterrestrial_marauders.py:253): hand its MT19937 state to the device
      # and write it back after every step.
      kind, key, pos = np.random.get_state()[:3]
      if kind != 'MT19937':
        raise RuntimeError('global NumPy RNG is not MT19937')
      rng_states = np.concatenate([key, [pos]]).astype(np.uint32)[None]
    self._batched = batched.BatchedEngine([lowered], batch=1, auto_reset=False,
                                          rng_states=rng_states)
    self._showtime = True
    self._chars = set(self._sprites_and_drapes) | set(self._backdrop.palette)
    return self._wrap(self._batched.its_showtime())

  def play(self, actions):
    """engine.py:583-639."""
    if not self._showtime:
      raise RuntimeError('play() cannot be called until the Engine is placed in "play '
                         'mode" via the its_showtime() method.')
    if self._game_over:
      raise RuntimeError('play() was called after the episode handled by this Engine '
                         'has terminated.')
    if self._batched.game.program == _lib.PROG_FIXTURE:
      return self._wrap(self._batched.play([self._fixture_row(actions)]))
    action = _lib.ACTION_NONE if actions is None else int(actions)
    return self._wrap(self._batched.play([action]))

  _MOTION_NAMES = ('n', 'ne', 'e', 'se', 's', 'sw', 'w', 'nw')

  def _fixture_row(self, actions):
    """General-program action row from the fixture conventions
    (tests/test_things.py:219-250): a direction string for everybody, or
    {char: direction}; unknown / missing = stay.  Directive keys '_reward',
    '_terminate', '_z' — or '_directives', an ordered list of Plot calls such as
    ('terminate_episode', 0.5) — stand in for post_update code injection."""
    from pycolab_b200.games import fixtures
    code = lambda d: self._MOTION_NAMES.index(d) if d in self._MOTION_NAMES else 8
    order = ''.join(self._batched.game.groups)
    if isinstance(actions, dict):
      motions = {ch: code(actions.get(ch)) for ch in order}
      return fixtures.action_rows(self._batched.game, motions, actions.get('_reward'),
                                  bool(actions.get('_terminate')), actions.get('_z'),
                                  directives=actions.get('_directives'))
    return fixtures.action_rows(self._batched.game, {ch: code(actions) for ch in order})

  def _wrap(self, result):
    import torch
    torch.cuda.synchronize(self._batched.device)
    board = result.board[0].cpu().numpy().copy()
    # d_reward is int32; games whose reference rewards are Python floats
    # (examples/classics) get the equal float back.
    reward = (self._batched.game.reward_type(int(result.reward[0]))
              if int(result.has_reward[0]) else None)
    discount = float(result.discount[0])
    self._game_over = bool(int(result.done[0]))
    self._sync_things()
    if self._batched.rng is not None:
      words = self._batched.rng[0].cpu().numpy().view(np.uint32)
      old = np.random.get_state()
      np.random.set_state((old[0], words[:624].copy(), int(words[624]), old[3], old[4]))
    errors = int(self._batched.error_codes()[0])
    if errors & _lib.ENV_ERR_ORDER_MISMATCH:
      raise RuntimeError('a scrolling order shares no component with the motion an '
                         'egocentric entity was to carry out in the same game iteration')
    if errors & _lib.ENV_ERR_EMPTY_CHOICE:
      raise ValueError("'a' cannot be empty unless no samples are taken")
    if errors & _lib.ENV_ERR_BAD_Z:
      raise RuntimeError('A z-order change directive named a Sprite or Drape that does '
                         'not exist')
    if errors & _lib.ENV_ERR_INDEX:
      raise IndexError('a board look-up fell off the array')
    if self._occlusion_in_layers:
      layers = rendering.LazyLayers(board, self._chars)
    else:
      # BaseUnoccludedObservationRenderer (rendering.py:187-301) on the device:
      # one kernel paints every character's un-occluded mask from the packed state.
      order = ''.join(sorted(self._chars))
      planes = self._batched.unoccluded_layers(order)[0].cpu().numpy()
      layers = {ch: planes[k] for k, ch in enumerate(order)}
    self._board = rendering.Observation(board=board, layers=layers)
    return self._board, reward, discount

  def _sync_things(self):
    """Mirror device records back into the entity objects (read-only peeking)."""
    b = self._batched
    sprites = b.sprites[0].cpu().numpy()
    drapes = b.drapes[0].cpu().numpy()
    self._the_plot._frame = int(b.plot[0, _lib.P_FRAME])
    if b.game.sync_plot is not None:       # dict entries the game keeps on the device
      b.game.sync_plot(self, b.plot[0].cpu().numpy())
    if b.game.backdrop_role == 'river':    # RiverBackdrop.update as a rotation count
      if self._backdrop_template is None:
        self._backdrop_template = self._backdrop.curtain.copy()
      r0, r1 = b.game.program_arg[1], b.game.program_arg[2]
      self._backdrop.curtain[r0:r1] = np.roll(self._backdrop_template[r0:r1],
                                              -int(b.plot[0, _lib.P_AUX0]), axis=1)
    if b.z_order is not None:             # Plot.change_z_order happened on the device
      order = [chr(c) for c in b.z_order[0].cpu().numpy()]
      self._sprites_and_drapes = collections.OrderedDict(
          (ch, self._sprites_and_drapes[ch]) for ch in order)
    for i, ch in enumerate(b.sprite_chars):
      ent, rec = self._sprites_and_drapes[ch], sprites[i]
      ent._position = things.Sprite.Position(int(rec[_lib.S_ROW]), int(rec[_lib.S_COL]))
      ent._visible = bool(rec[_lib.S_FLAGS] & 1)
      if isinstance(ent, prefab_sprites.MazeWalker):
        ent._virtual_row, ent._virtual_col = int(rec[_lib.S_VROW]), int(rec[_lib.S_VCOL])
    if b.game.program == _lib.PROG_BOX_WORLD:
      # the keys, locks and gem live in one cell plane; the player counts its moves
      chars = b.plane()[0, :, :self._cols].cpu().numpy() & 0x7f
      for ch, ent in self._sprites_and_drapes.items():
        if isinstance(ent, things.Drape):
          np.copyto(ent.curtain, chars == ord(ch))
      self._sprites_and_drapes[b.sprite_chars[0]]._step_counter = int(sprites[0, _lib.S_AUX0])
    for i, ch in enumerate(b.drape_chars):
      ent, rec = self._sprites_and_drapes[ch], drapes[i]
      if isinstance(ent, prefab_drapes.Scrolly):
        ent._northwest_corner = things.Sprite.Position(int(rec[_lib.D_CORNER_R]),
                                                       int(rec[_lib.D_CORNER_C]))
        # registers behind pattern_position_prescroll / _postscroll (drapes.py:378-441)
        ent._prescroll_northwest_corner = things.Sprite.Position(int(rec[_lib.D_PRE_R]),
                                                                 int(rec[_lib.D_PRE_C]))
        last = int(rec[_lib.D_LAST_FRAME])
        ent._last_maybe_move_frame = -float('inf') if last == _lib.NEVER else last
        if b.game.pattern_mutable.get(i):      # e.g. coins picked up on the device
          from pycolab_b200 import lowering
          packed = b.patterns[i][0].cpu().numpy().view(np.uint32)
          np.copyto(ent.whole_pattern, lowering.unpack_rows(packed, ent.whole_pattern.shape[1]))
      np.copyto(ent.curtain, b.curtain(ch)[0].cpu().numpy())
      if b.game.program == _lib.PROG_APERTURE:       # ApertureDrape._apertures
        cells = [int(rec[_lib.D_AUX0]), int(rec[_lib.D_AUX1])]
        ent._apertures = [None if c < 0 else (c >> 16, c & 0xffff) for c in cells]

  # ------------------------------------------------------------ properties
  @property
  def the_plot(self):
    return self._the_plot

  @property
  def rows(self):
    return self._rows

  @property
  def cols(self):
    return self._cols

  @property
  def game_over(self):
    return self._game_over

  @property
  def z_order(self):
    return list(self._sprites_and_drapes.keys())

  @property
  def backdrop(self):
    return self._backdrop

  @property
  def things(self):
    return dict(self._sprites_and_drapes)

  @property
  def batched(self):
    """The underlying batch-1 `BatchedEngine` (after its_showtime())."""
    return self._batched

  # -------------------------------------------------------------- helpers
  def _no_showtime(self, method_name):
    if self._showtime:
      raise RuntimeError('{} should not be called after its_showtime() has been '
                         'called'.format(method_name))

  def _check_unclaimed(self, characters):
    for char in characters:
      if self._backdrop and char in self._backdrop.palette:
        raise RuntimeError('Character {!r} is already being used by the '
                           'backdrop'.format(char))
      if char in self._sprites_and_drapes:
        raise RuntimeError('Character {!r} is already being used by a sprite or a '
                           'drape'.format(char))

  def _check_chars(self, characters, mandatory_len=None):
    if mandatory_len is not None and len(characters) != mandatory_len:
      raise ValueError('{!r}, a string of length {}, was used where a string of length '
                       '{} was required'.format(characters, len(characters),
                                                mandatory_len))
    for char in characters:
      try:
        ord(char)
      except TypeError:
        raise ValueError('Character {} is not an ASCII character'.format(char))


class Palette(object):
  """Legal backdrop characters with attribute access (engine.py:877-986):
  `palette.a` -> ord('a'), plus spelled-out aliases for punctuation/digits."""

  _ALIASES = {}
  for _names, _ch in (
      ('backtick backquote grave', '`'), ('tilde', '~'), ('zero', '0'), ('one', '1'),
      ('two', '2'), ('three', '3'), ('four', '4'), ('five', '5'), ('six', '6'),
      ('seven', '7'), ('eight', '8'), ('nine', '9'),
      ('bang exclamation exclamation_point exclamation_pt', '!'), ('at', '@'),
      ('hash hashtag octothorpe number_sign pigpen pound', '#'),
      ('dollar dollar_sign buck mammon', '$'), ('percent percent_sign food', '%'),
      ('carat circumflex trap', '^'), ('and_sign ampersand', '&'),
      ('asterisk star splat', '*'), ('lbracket left_bracket lparen left_paren', '('),
      ('rbracket right_bracket rparen right_paren', ')'), ('dash hyphen', '-'),
      ('underscore', '_'), ('plus add', '+'), ('equal equals', '='),
      ('lsquare left_square_bracket', '['), ('rsquare right_square_bracket', ']'),
      ('lbrace lcurly left_brace left_curly left_curly_brace', '{'),
      ('rbrace rcurly right_brace right_curly right_curly_brace', '}'),
      ('pipe bar', '|'), ('backslash back_slash reverse_solidus', '\\'),
      ('semicolon', ';'), ('colon', ':'), ('tick quote inverted_comma prime', "'"),
      ('quotes double_inverted_commas quotation_mark', '"'), ('zed', 'z'),
      ('comma', ','), ('less_than langle left_angle left_angle_bracket', '<'),
      ('period full_stop', '.'),
      ('greater_than rangle right_angle right_angle_bracket', '>'),
      ('question question_mark', '?'), ('slash solidus', '/')):
    for _name in _names.split():
      _ALIASES[_name] = _ch
  del _names, _ch, _name

  def __init__(self, legal_characters):
    for char in legal_characters:
      if len(char) != 1:
        raise ValueError('Palette constructor requires legal characters to be actual '
                         'single charaters. "{}" is not.'.format(char))
    self._legal_characters = set(legal_characters)

  def __getattr__(self, name):
    if name.startswith('__') or name == '_legal_characters':
      raise AttributeError(name)          # copy/pickle probes before __init__
    return self._lookup(name, AttributeError)

  def __getitem__(self, key):
    return self._lookup(key, IndexError)

  def __contains__(self, key):
    return key in self._legal_characters

  def __iter__(self):
    return iter(self._legal_characters)

  def __getstate__(self):
    return self._legal_characters

  def __setstate__(self, state):
    self._legal_characters = set(state)

  def _lookup(self, key, error):
    key = self._ALIASES.get(key, key)
    if key in self._legal_characters:
      return ord(key)
    raise error('{} is not a legal character in this Palette; legal characters are '
                '{}.'.format(key, list(self._legal_characters)))
