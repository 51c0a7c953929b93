"""CPU tests of the host side: C-ABI library surface, facade set-up API,
lowering, compat loading of example modules."""

import os
import sys
import re

import numpy as np
import pytest

import golden_cases as gc
import reference_trace as rt
import trajectory as tj
from oracle import games as ogames
from pycolab_b200 import _lib
from pycolab_b200 import ascii_art
from pycolab_b200 import engine as engine_mod
from pycolab_b200 import levels
from pycolab_b200 import lowering
from pycolab_b200 import things
from pycolab_b200.errors import DeviceOnlyError, NotLoweredError
from pycolab_b200.games import extraterrestrial_marauders as g_marauders
from pycolab_b200.games import scrolly_maze as g_scrolly
from pycolab_b200.games import warehouse_manager as g_warehouse
from pycolab_b200.prefab_parts import sprites as prefab_sprites

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------ C-ABI library

def _header_functions():
  text = open(os.path.join(ROOT, 'include', 'pcl.h')).read()
  text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
  return sorted(set(re.findall(r'\b(pcl_[a-z_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
  import ctypes
  assert os.path.exists(_lib.LIB_PATH), 'build libpcl.so first (__graft_entry__.build)'
  lib = ctypes.CDLL(_lib.LIB_PATH)
  declared = _header_functions()
  assert len(declared) >= 14
  for name in declared:
    assert hasattr(lib, name), name
  assert sorted(_lib.SYMBOLS) == declared


def test_binding_loads_and_reports_abi():
  lib = _lib.load()
  assert lib.pcl_abi_version() == _lib.ABI_VERSION
  assert _lib.status_string(_lib.ERR_UNSUPPORTED) == 'game not lowered to a device program'


def test_binding_structs_match_the_header():
  """The library reports sizeof() of every struct that crosses the boundary;
  `_lib.load()` refuses a binding whose ctypes layouts disagree."""
  import ctypes as C
  lib = _lib.load()
  sizes = (C.c_int32 * 4)()
  assert lib.pcl_struct_sizes(sizes) == _lib.OK
  assert list(sizes) == [C.sizeof(_lib.Spec), C.sizeof(_lib.State), C.sizeof(_lib.Outputs),
                         C.sizeof(_lib.CropSpec)]


def test_create_rejects_bad_specs_without_gpu():
  import ctypes as C
  lib = _lib.load()
  h = C.c_void_p()
  spec = _lib.Spec()
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(h)) == _lib.ERR_INVALID  # abi 0
  spec.abi_version = _lib.ABI_VERSION
  spec.rows, spec.cols, spec.pitch = 10, 30, 30                              # pitch % 16
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(h)) == _lib.ERR_INVALID
  spec.pitch = 32
  spec.program = 99
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(h)) == _lib.ERR_UNSUPPORTED
  spec.program = _lib.PROG_NONE
  assert lib.pcl_create(C.byref(spec), 4, -1, C.byref(h)) == _lib.OK
  out = _lib.Outputs()
  assert lib.pcl_step(h, None, C.byref(out), None) == _lib.ERR_UNBOUND
  assert lib.pcl_destroy(h) == _lib.OK


def _create(spec, batch=4):
  import ctypes as C
  lib = _lib.load()
  h = C.c_void_p()
  status = lib.pcl_create(C.byref(spec), batch, -1, C.byref(h))   # device -1: no CUDA call
  if status == _lib.OK:
    lib.pcl_destroy(h)
  return status


def test_every_lowered_game_passes_create_validation_without_gpu():
  """lowering -> pcl_spec -> pcl_create's validation, for one level of every
  device program (no GPU needed: device = -1 skips cudaSetDevice)."""
  import importlib
  import golden_cases as gc
  import trajectory as tj
  from pycolab_b200.games import aperture, better_scrolly_maze, fluvial_natation
  games = [g_scrolly.make_game(*levels.scrolly_maze_level(0, world_shape=(33, 33),
                                                          board_shape=(16, 16))),
           g_warehouse.make_game(levels.warehouse_level(1), ' '),
           g_marauders.make_game(levels.marauders_level()),
           better_scrolly_maze.make_game(tj.u8_to_art(gc.load('better_stock_L0')['art'])),
           fluvial_natation.make_game(), aperture.make_game(levels.aperture_level())]
  for kind in ('four_rooms', 'cliff_walk', 'chain_walk'):
    mod = importlib.import_module('pycolab_b200.games.classics.' + kind)
    games += [mod.make_game(), mod.make_game(levels.classic_level(kind))]
  programs = set()
  for game in games:
    lowered = lowering.lower(game)
    programs.add(lowered.program)
    assert _create(lowered.make_spec(auto_reset=True)) == _lib.OK, lowered.program
  assert programs == {_lib.PROG_SCROLLY_MAZE, _lib.PROG_WAREHOUSE, _lib.PROG_MARAUDERS,
                      _lib.PROG_BETTER_SCROLLY, _lib.PROG_CLASSICS, _lib.PROG_APERTURE}


def test_create_rejects_malformed_specs_of_the_newer_programs():
  from pycolab_b200.games import aperture, fluvial_natation
  from pycolab_b200.games.classics import four_rooms
  spec = lowering.lower(four_rooms.make_game()).make_spec(True)
  spec.program_arg[0] = 9                                   # unknown rule set
  assert _create(spec) == _lib.ERR_INVALID
  spec = lowering.lower(fluvial_natation.make_game()).make_spec(True)
  spec.impassable[0][1] = 1 << 3                            # a swimmer that reads the board ('#')
  assert _create(spec) == _lib.ERR_UNSUPPORTED
  spec = lowering.lower(aperture.make_game(levels.aperture_level())).make_spec(True)
  spec.z_order[0], spec.z_order[1] = spec.z_order[1], spec.z_order[0]   # player under the drape
  assert _create(spec) == _lib.ERR_UNSUPPORTED
  spec = lowering.lower(aperture.make_game(levels.aperture_level())).make_spec(True)
  spec.n_groups, spec.group_len[0], spec.group_len[1] = 1, 2, 0         # one update group
  assert _create(spec) == _lib.ERR_UNSUPPORTED
  spec = lowering.lower(four_rooms.make_game()).make_spec(True)
  assert _create(spec, batch=0) == _lib.ERR_INVALID


def test_missing_library_fails_loudly(monkeypatch):
  monkeypatch.setattr(_lib, '_lib', None)
  monkeypatch.setattr(_lib, 'LIB_PATH', '/nonexistent/libpcl.so')
  with pytest.raises(_lib.PclLibraryError):
    _lib.load()


def test_no_cpu_path():
  import torch
  if torch.cuda.is_available():
    pytest.skip('GPU present')
  from pycolab_b200 import batched
  art = levels.scrolly_maze_level(0, world_shape=(33, 33), board_shape=(16, 16))
  with pytest.raises(_lib.PclLibraryError):
    batched.BatchedEngine([g_scrolly.make_game(*art)], batch=2)
  with pytest.raises(_lib.PclLibraryError):
    g_scrolly.make_game(*art).its_showtime()


# ----------------------------------------------------------------- lowering

def test_pack_rows_round_trip():
  rs = np.random.RandomState(0)
  for cols in (1, 31, 32, 33, 64, 89, 129):
    mask = rs.random_sample((7, cols)) < 0.4
    words = (cols + 31) // 32 + 1
    packed = lowering.pack_rows(mask, words)
    assert packed.shape == (7, words) and packed.dtype == np.uint32
    np.testing.assert_array_equal(lowering.unpack_rows(packed, cols), mask)
    assert not packed[:, -1].any()
    c = cols - 1
    assert bool((packed[3, c >> 5] >> (c & 31)) & 1) == bool(mask[3, c])


def _check_sprites(game, world, chars):
  for i, ch in enumerate(chars):
    w, rec = world.things[ch], game.sprites[i]
    assert tuple(rec[:4]) == (w.row, w.col, w.vrow, w.vcol), ch
    assert bool(rec[_lib.S_FLAGS] & 1) == bool(w.visible), ch
    prior = (rec[_lib.S_FLAGS] >> 1) & 3
    assert {0: None, 1: False, 2: True}[prior] == w.prior_visible, ch


@pytest.mark.parametrize('name', ['scrolly_stock_L0', 'scrolly_stock_L2', 'scrolly_gen64_s0'])
def test_lower_scrolly_matches_oracle_initial_state(name):
  g = gc.load(name)
  maze, board, beneath = gc.scrolly_art(g)
  game = lowering.lower(g_scrolly.make_game(maze, board, beneath))
  world = ogames.make_scrolly_maze(maze, board, '+', beneath)
  assert game.program == _lib.PROG_SCROLLY_MAZE
  assert (game.rows, game.cols) == (world.rows, world.cols)
  assert game.pitch % 16 == 0 and game.pitch >= game.cols
  assert game.sprite_chars == 'Pabc' and game.drape_chars == '#@'
  assert game.z_order == 'abc@#P' and game.groups == ['#', 'abcP', '@']
  _check_sprites(game, world, 'Pabc')
  for d, ch in enumerate('#@'):
    np.testing.assert_array_equal(
        lowering.unpack_rows(game.patterns[d], game.pattern_cols), world.things[ch].pattern)
    assert tuple(game.drapes[d][:2]) == world.things[ch].corner
    assert game.margins[d] == (2, 3)
  assert game.plot[_lib.P_AUX0] == world.things['@'].pattern.sum()
  assert game.plot[_lib.P_FRAME] == -1
  np.testing.assert_array_equal(game.backdrop[:, :game.cols], world.backdrop)
  assert [int(game.sprites[i][_lib.S_AUX0]) for i in (1, 2, 3)] == [
      int(world.things[c].aux['moving_east']) for c in 'abc']
  assert game.egocentric == [True, False, False, False]


@pytest.mark.parametrize('name', ['warehouse_stock_L0', 'warehouse_stock_L1',
                                  'warehouse_gen80_s3'])
def test_lower_warehouse_matches_oracle_initial_state(name):
  g = gc.load(name)
  art, wlb = gc.warehouse_art(g)
  game = lowering.lower(g_warehouse.make_game(art, wlb))
  world = ogames.make_warehouse(art, wlb)
  chars = bytes(g['sprite_chars']).decode()
  assert game.program == _lib.PROG_WAREHOUSE and game.sprite_chars == chars
  _check_sprites(game, world, chars)
  np.testing.assert_array_equal(game.backdrop[:, :game.cols], world.backdrop)
  for i, ch in enumerate(chars):
    want = lowering.char_set_mask(chr(c) for c in world.things[ch].impassable)
    assert game.impassable[i] == want


def test_lower_marauders_matches_oracle_initial_state():
  art = levels.marauders_level()
  game = lowering.lower(g_marauders.make_game(art))
  world = ogames.make_marauders(art, np.random.RandomState(0))
  assert game.program == _lib.PROG_MARAUDERS and game.needs_rng
  _check_sprites(game, world, 'Pabcdyz')
  for d, ch in enumerate('BX'):
    np.testing.assert_array_equal(lowering.unpack_rows(game.bits[d], game.cols),
                                  world.things[ch].curtain)
  assert game.drapes[1][_lib.D_AUX0] == -1
  assert game.confined == [True] + [False] * 6
  # bolts start hidden off-board with their visibility stashed (sprites.py:223-249)
  assert all(game.sprites[i][_lib.S_FLAGS] == 4 for i in range(1, 7))


def test_unknown_entity_class_is_refused():
  class Wanderer(prefab_sprites.MazeWalker):
    def __init__(self, corner, position, character):
      super(Wanderer, self).__init__(corner, position, character, impassable='#')

    def update(self, actions, board, layers, backdrop, things, the_plot):
      self._north(board, the_plot)

  game = ascii_art.ascii_art_to_game(['#####', '# w #', '#####'], ' ', {'w': Wanderer})
  with pytest.raises(NotLoweredError):
    lowering.lower(game)
  with pytest.raises(NotLoweredError):
    game.its_showtime()
  with pytest.raises(DeviceOnlyError):
    game.things['w']._north(None, None)


def test_overriding_update_of_a_lowered_class_is_refused():
  class Cheater(g_scrolly.PlayerSprite):
    def update(self, actions, board, layers, backdrop, things, the_plot):
      pass
  assert lowering.role_of.__name__ == 'role_of'
  corner = things.Sprite.Position(5, 5)
  with pytest.raises(NotLoweredError):
    lowering.role_of(Cheater(corner, things.Sprite.Position(1, 1), 'P', (1, 1)))


# ----------------------------------------------- facade set-up API behaviour

def test_engine_setup_errors_match_reference_contract():
  eng = engine_mod.Engine(3, 4)
  with pytest.raises(TypeError):
    eng.add_sprite('a', (0, 0), object)
  with pytest.raises(ValueError):
    eng.add_sprite('a', (5, 0), g_warehouse.PlayerSprite)
  eng.add_sprite('a', (1, 1), g_warehouse.PlayerSprite)
  with pytest.raises(RuntimeError):
    eng.add_sprite('a', (1, 2), g_warehouse.PlayerSprite)
  with pytest.raises(ValueError):
    eng.add_sprite('ab', (1, 2), g_warehouse.PlayerSprite)
  with pytest.raises(ValueError):
    eng.set_z_order('ab')
  with pytest.raises(RuntimeError):
    eng.play(0)
  eng.set_prefilled_backdrop(' #', np.full((3, 4), 32, np.uint8), things.Backdrop)
  with pytest.raises(RuntimeError):
    eng.set_backdrop(' ', things.Backdrop)
  assert eng.backdrop.palette.hash == ord('#')
  assert eng.backdrop.palette[' '] == 32
  with pytest.raises(AttributeError):
    eng.backdrop.palette.at


def test_ascii_art_errors():
  with pytest.raises(TypeError):
    ascii_art.ascii_art_to_uint8_nparray([['a', 'b'], ['c', 'd']])
  with pytest.raises(ValueError):
    ascii_art.ascii_art_to_uint8_nparray(['ab', 'c'])
  with pytest.raises(ValueError):
    ascii_art.ascii_art_to_game(['P '], ' ', {'P': g_warehouse.PlayerSprite},
                                update_schedule=[['Q']])
  with pytest.raises(ValueError):
    ascii_art.ascii_art_to_game(['PP'], ' ', {'P': g_warehouse.PlayerSprite})
  with pytest.raises(TypeError):
    ascii_art.Partial(int)


def test_maze_walker_constructor_contract():
  corner = things.Sprite.Position(4, 4)
  class Plain(prefab_sprites.MazeWalker):
    def update(self, *args):
      pass
  with pytest.raises(ValueError):
    Plain(corner, things.Sprite.Position(0, 0), 'x', 'x#')
  with pytest.raises(TypeError):
    Plain(corner, things.Sprite.Position(0, 0), 'x', [1, 2])
  bolt = g_marauders.UpwardLaserBoltSprite(corner, things.Sprite.Position(2, 2), 'a')
  assert bolt.position == (0, 0) and not bolt.visible and not bolt.on_the_board
  assert bolt.virtual_position == (-1, -1) and bolt._prior_visible is True
  bolt._teleport((3, 1))
  assert bolt.position == (3, 1) and bolt.visible


# ------------------- the original's example files, as they lower through compat
# tests/golden/reference_lowerings.json holds a digest of what each of the
# original's example files lowered to when loaded unmodified through `compat`
# (tests/golden/make_reference_traces.py); this package's twins must lower to
# exactly that.

@pytest.fixture
def compat_loader(tmp_path):
  """Writes a module source into tmp_path and loads it through `compat`, the way
  a user's copy of an example file is loaded."""
  from pycolab_b200 import compat
  saved = {k: v for k, v in sys.modules.items()
           if k == 'pycolab' or k.startswith('pycolab.')}
  compat.uninstall()
  compat.install()

  def load(name, source, copy='a'):
    path = tmp_path / copy / (name + '.py')
    path.parent.mkdir(exist_ok=True)
    path.write_text(source)
    return compat.load_example(str(path))
  yield load
  compat.uninstall()
  sys.modules.update(saved)


def test_reference_scrolly_maze_example_loads_and_lowers():
  for level in (0, 1, 2):
    maze, board, beneath = gc.scrolly_art(gc.load('scrolly_stock_L%d' % level))
    rt.check_lowering('scrolly_maze_%d' % level,
                      lowering.lower(g_scrolly.make_game(maze, board, beneath)))


def _user_copy_of_the_scrolly_maze_twin():
  """This package's scrolly_maze set-up as a user's module: imports through the
  `pycolab` alias, so its classes are not trusted by module."""
  import inspect
  return inspect.getsource(g_scrolly).replace('from pycolab_b200 import', 'from pycolab import') \
      .replace('from pycolab_b200.prefab_parts', 'from pycolab.prefab_parts')


def test_edited_copy_of_an_example_is_refused_not_replaced(compat_loader, monkeypatch):
  """A user's copy of scrolly_maze.py lowers while its classes are token-for-token
  the known implementation; with an edited class body the class is named like a
  lowered class but is NOT that class: NotLoweredError, never the stock kernel
  (lowering._is_known_implementation).  The known fingerprints are those of the
  original's classes; here they are pointed at the copy's own classes."""
  import inspect
  from pycolab_b200 import _fingerprints
  maze, board, beneath = gc.scrolly_art(gc.load('scrolly_stock_L0'))
  src = _user_copy_of_the_scrolly_maze_twin()
  mod = compat_loader('scrolly_maze', src)
  assert mod.PlayerSprite.__mro__[1] is prefab_sprites.MazeWalker   # `pycolab` is this package
  with pytest.raises(NotLoweredError, match='source differs'):
    lowering.lower(mod.make_game(maze, board, beneath))     # not the original's source
  for name in ('PlayerSprite', 'PatrollerSprite', 'MazeDrape', 'CashDrape'):
    monkeypatch.setitem(_fingerprints.KNOWN, ('scrolly_maze', name),
                        lowering.source_fingerprint(inspect.getsource(getattr(mod, name))))
  same = compat_loader('scrolly_maze', '# my copy\n' + src.replace('\n\n', '\n\n\n', 1)
                       .replace('\nclass PlayerSprite', '\n# the explorer\nclass PlayerSprite'),
                       copy='same')
  rt.check_lowering('scrolly_maze_0', lowering.lower(same.make_game(maze, board, beneath)))
  assert "impassable='#')" in src
  edited = compat_loader('scrolly_maze', src.replace("impassable='#')", "impassable='#@')", 1),
                         copy='edited')
  with pytest.raises(NotLoweredError, match='source differs'):
    lowering.lower(edited.make_game(maze, board, beneath))


_FINGERPRINTED = '''class PlayerSprite(prefab_sprites.MazeWalker):
  """A walker that goes north on action 0 and stays put otherwise."""

  def update(self, actions, board, layers, backdrop, things, the_plot):
    del backdrop, things  # unused
    if actions == 0:
      self._north(board, the_plot)
    else:
      self._stay(board, the_plot)
'''


def test_source_fingerprint_normalisation_is_pinned():
  """_fingerprints.KNOWN holds source_fingerprint() of the original's classes, so
  the normalisation must not drift: a change to it would refuse every user's
  unmodified example file.  Comments, blank lines, indentation width and an
  enclosing indent do not count; any token does."""
  import textwrap
  want = '231bf765e8f4715d643edcbd053c360c919d3e6aac35755d51e45a5d09621e4f'
  assert lowering.source_fingerprint(_FINGERPRINTED) == want
  reindented = textwrap.indent(_FINGERPRINTED.replace('  ', '    '), '    ')
  commented = _FINGERPRINTED.replace('\n\n', '\n\n  # the update\n\n').replace(
      'actions == 0:', 'actions == 0:  # north')
  assert lowering.source_fingerprint(reindented) == want
  assert lowering.source_fingerprint(commented) == want
  for edit in [('_north', '_south'), ('== 0', '== 1'), ('otherwise', 'always'),
               ('del backdrop, things  # unused', 'del backdrop, things, layers')]:
    assert lowering.source_fingerprint(_FINGERPRINTED.replace(*edit)) != want, edit


def test_reference_warehouse_example_loads_and_lowers():
  for level in (0, 1, 2):
    art, wlb = gc.warehouse_art(gc.load('warehouse_stock_L%d' % level))
    rt.check_lowering('warehouse_manager_%d' % level,
                      lowering.lower(g_warehouse.make_game(art, wlb)))


def test_reference_marauders_example_loads_and_lowers():
  rt.check_lowering('extraterrestrial_marauders',
                    lowering.lower(g_marauders.make_game(levels.marauders_level())))


def test_reference_example_outside_the_lowered_set_is_refused(compat_loader):
  # a game whose entities carry their own Python update() (tennis, or anything a
  # user writes) has no device program
  mod = compat_loader('tennnnnnnnnnnnnnnnnnnnnnnnis', """
from pycolab import ascii_art
from pycolab import things


class BallSprite(things.Sprite):
  def update(self, actions, board, layers, backdrop, things, the_plot):
    self._position = self.Position(self.position.row, (self.position.col + 1) % 5)


def make_game():
  return ascii_art.ascii_art_to_game(['  o  '], ' ', sprites={'o': BallSprite})
""")
  with pytest.raises(NotLoweredError):
    lowering.lower(mod.make_game())


def test_reference_better_scrolly_example_loads_and_lowers():
  from pycolab_b200.games import better_scrolly_maze as g_better
  for level in (0, 1, 2):
    art = [bytes(r).decode('ascii') for r in gc.load('better_stock_L%d' % level)['art']]
    ours = lowering.lower(g_better.make_game(art))
    assert ours.program == _lib.PROG_BETTER_SCROLLY
    rt.check_lowering('better_scrolly_maze_%d' % level, ours)
  # the example's croppers are this package's classes
  views = g_better.make_croppers()
  assert [type(v).__name__ for v in views] == ['ScrollingCropper', 'ScrollingCropper',
                                               'FixedCropper']


@pytest.mark.parametrize('kind', ['four_rooms', 'cliff_walk', 'chain_walk'])
def test_reference_classics_examples_load_and_lower(kind):
  import importlib
  from oracle import games as ogames
  ours_mod = importlib.import_module('pycolab_b200.games.classics.' + kind)
  ours = lowering.lower(ours_mod.make_game())
  assert ours.program == _lib.PROG_CLASSICS and ours.reward_type is float
  rt.check_lowering(kind, ours)
  # ... and the lowered initial state is the oracle's
  world = ogames.make_classic(kind, list(ours_mod.GAME_ART))
  w = world.things['P']
  assert tuple(ours.sprites[0, :5]) == (w.row, w.col, w.vrow, w.vcol, 1)
  np.testing.assert_array_equal(ours.backdrop[:, :ours.cols], world.backdrop)
  assert bool(ours.confined[0]) == w.confined


def test_reference_aperture_example_loads_and_lowers():
  from pycolab_b200.games import aperture as ours_mod
  for level in (0, 1, 2):
    art = [bytes(r).decode('ascii') for r in gc.load('aperture_stock_L%d' % level)['art']]
    ours = lowering.lower(ours_mod.make_game(art))
    assert ours.program == _lib.PROG_APERTURE
    assert list(ours.drapes[0, [_lib.D_AUX0, _lib.D_AUX1]]) == [-1, -1]
    rt.check_lowering('aperture_%d' % level, ours)


def test_reference_fluvial_natation_loads_and_lowers():
  """A Backdrop subclass with update() logic is lowered with its own game only."""
  from pycolab_b200.games import fluvial_natation as ours_mod
  from pycolab_b200.games.classics import four_rooms
  ours = lowering.lower(ours_mod.make_game())
  assert ours.program == _lib.PROG_CLASSICS and ours.backdrop_role == 'river'
  assert list(ours.program_arg[:3]) == [_lib.CLASSIC_FLUVIAL, 1, 4] and ours.reward_type is int
  rt.check_lowering('fluvial_natation', ours)
  # the river under another game's entities is refused, and so is an unknown Backdrop
  with pytest.raises(NotLoweredError):
    lowering.lower(ascii_art.ascii_art_to_game(four_rooms.GAME_ART, ' ',
                                               sprites={'P': four_rooms.PlayerSprite},
                                               backdrop=ours_mod.RiverBackdrop))

  class Odd(ours_mod.RiverBackdrop):
    def update(self, *args, **kwargs):
      pass
  with pytest.raises(NotLoweredError):
    lowering.lower(ascii_art.ascii_art_to_game(ours_mod.GAME_ART, ' ',
                                               sprites={'P': ours_mod.PlayerSprite},
                                               backdrop=Odd))


def test_reference_test_fixtures_load_and_lower():
  """The original's tests/test_things.py fixtures lowered to the general device
  program exactly as this package's games/fixtures.py does."""
  from pycolab_b200.games import fixtures
  kw, cfg = gc.fixture_kwargs(gc.load('fixture_scrolly_0'))
  ours = lowering.lower(fixtures.make_game(kw['art'], ' ', kw['walkers'], kw['scrollys'], '',
                                           kw['update_schedule'], kw['z_order']))
  assert ours.program == _lib.PROG_FIXTURE and ours.dynamic_z
  assert ours.drape_kind == [1, 1]
  rt.check_lowering('test_things_fixture_scrolly_0', ours)


def test_reference_host_only_unit_tests_pass_against_this_package():
  """What the original's host-only unit tests (ascii_art_test.py,
  scrolling_test.py::testProtocol) check, on this package: malformed art is
  refused with messages that say what was wrong (and so are malformed entity
  tables), and the scrolling-protocol helpers register
  participants per group, grant motions for the next frame only, accept one
  order per frame and name the offending entity in their errors."""
  from pycolab_b200 import plot as plot_lib
  from pycolab_b200.protocols import scrolling

  class Walker(things.Sprite):
    def update(self, *args, **kwargs):
      pass

  class Curtain(things.Drape):
    def update(self, *args, **kwargs):
      pass

  # ascii_art_to_uint8_nparray: ragged rows, a row that is not a string, rows of
  # single characters
  with pytest.raises(ValueError, match='must be a list'):
    ascii_art.ascii_art_to_uint8_nparray(['ab', 'abc'])
  with pytest.raises(TypeError, match='must be a list'):
    ascii_art.ascii_art_to_uint8_nparray(['ab', 12])
  with pytest.raises(TypeError, match='Did you pass a list of list of single characters'):
    ascii_art.ascii_art_to_uint8_nparray([['a', 'b'], ['c', 'd']])
  # ascii_art_to_game: ragged art, a character that is both sprite and drape, a
  # sprite character appearing twice
  with pytest.raises(ValueError):
    ascii_art.ascii_art_to_game(['P ', ' '], ' ', {'P': Walker})
  with pytest.raises(RuntimeError, match='already being used'):
    ascii_art.ascii_art_to_game(['P '], ' ', {'P': Walker}, {'P': Curtain})
  with pytest.raises(ValueError):
    ascii_art.ascii_art_to_game(['PP'], ' ', {'P': Walker})

  sprite = Walker(things.Sprite.Position(6, 7), things.Sprite.Position(2, 3), 'P')
  drape = Curtain(np.zeros((6, 7), dtype=bool), 'X')
  the_plot = plot_lib.Plot()
  for who in (sprite, drape):
    scrolling.participate_as_egocentric(who, the_plot, scrolling_group='g')
  assert scrolling.egocentric_participants(drape, the_plot, scrolling_group='g') == {sprite, drape}
  assert scrolling.get_order(sprite, the_plot, scrolling_group='g') is None
  with pytest.raises(scrolling.Error, match="known to belong to scrolling group 'g'"):
    scrolling.get_order(sprite, the_plot, scrolling_group='h')
  with pytest.raises(TypeError):
    scrolling.participate_as_egocentric(object(), the_plot)

  the_plot = plot_lib.Plot()
  for who in (sprite, drape):
    scrolling.participate_as_egocentric(who, the_plot)
  for frame in range(8):                       # the frame counter advances one at a time
    the_plot.frame = frame
  scrolling.permit(sprite, the_plot, motions=[(0, 0), (0, -1), (-1, 0)])
  scrolling.permit(drape, the_plot, motions=[(0, 0), (-1, 0)])
  assert not any(scrolling.is_possible(drape, the_plot, m) for m in [(0, 0), (-1, 0)])
  the_plot.frame = 8                           # permits hold for the next frame only
  assert scrolling.is_possible(sprite, the_plot, (0, 0))
  assert scrolling.is_possible(sprite, the_plot, (-1, 0))
  assert not scrolling.is_possible(sprite, the_plot, (0, -1))   # the drape never allowed it
  with pytest.raises(scrolling.Error, match="impossible scrolling motion"):
    scrolling.order(drape, the_plot, (0, -1))
  scrolling.order(drape, the_plot, (-1, 0))
  assert scrolling.get_order(sprite, the_plot) == (-1, 0)
  with pytest.raises(scrolling.Error, match="Sprite or Drape handling character 'P'.*second"):
    scrolling.order(sprite, the_plot, (0, 0))
  the_plot.frame = 9
  assert scrolling.get_order(sprite, the_plot) is None
  assert not scrolling.is_possible(sprite, the_plot, (0, 0))    # permits expired


@pytest.mark.parametrize('call', [lambda p: p.add_reward(1), lambda p: p.terminate_episode(),
                                  lambda p: p.change_default_discount(0.5),
                                  lambda p: p.change_z_order('P', None)])
def test_plot_directives_before_showtime_are_refused(call):
  """engine.py:761-847 folds whatever the Plot holds into frame 0; the device's frame 0
  starts from clean directives, so the facade refuses instead of dropping them."""
  art = levels.scrolly_maze_level(3, world_shape=(33, 33), board_shape=(16, 16))
  game = g_scrolly.make_game(*art)
  call(game.the_plot)
  with pytest.raises(NotLoweredError, match='before its_showtime'):
    game.its_showtime()


def _bound_handle(game, batch=4):
  """A handle created and BOUND on the CPU: pcl_bind_state only records pointers, so
  made-up non-null addresses are enough to reach the argument checks of the entry
  points behind it (nothing is launched)."""
  import ctypes as C
  lib = _lib.load()
  handle = C.c_void_p()
  spec = game.make_spec(True)
  assert lib.pcl_create(C.byref(spec), batch, -1, C.byref(handle)) == _lib.OK
  st = _lib.State()
  fake = 0x10000
  for name in ('d_backdrop', 'd_sprites', 'd_sprites_init', 'd_drapes', 'd_drapes_init',
               'd_plot', 'd_plot_init'):
    setattr(st, name, fake)
  for d in range(2):
    st.d_pattern[d], st.d_pattern_init[d] = fake, fake
    st.pattern_bstride[d], st.pattern_init_bstride[d] = 64, 64
  assert lib.pcl_bind_state(handle, C.byref(st)) == _lib.OK
  return lib, handle


def test_attach_cropper_argument_checks_on_cpu():
  """pcl_attach_cropper: unbound handle, bad window, drape tracking, programs without
  the epilogue, detach — all decided before anything touches the device."""
  import ctypes as C
  from pycolab_b200 import batched
  art = levels.scrolly_maze_level(3, world_shape=(33, 33), board_shape=(16, 16))
  game = lowering.lower(g_scrolly.make_game(*art))
  lib = _lib.load()
  raw = C.c_void_p()
  spec0 = game.make_spec(True)
  assert lib.pcl_create(C.byref(spec0), 4, -1, C.byref(raw)) == _lib.OK
  crop = batched.scrolling_crop_spec(5, 5, 0, pad_char=' ', scroll_margins=(None, None))
  assert lib.pcl_attach_cropper(raw, C.byref(crop), 0x20000, 0x30000) == _lib.ERR_UNBOUND
  lib.pcl_destroy(raw)

  lib, h = _bound_handle(game)
  assert lib.pcl_attach_cropper(h, C.byref(crop), 0x20000, 0x30000) == _lib.OK
  assert lib.pcl_attach_cropper(h, C.byref(crop), None, 0x30000) == _lib.ERR_INVALID
  assert lib.pcl_attach_cropper(h, None, None, None) == _lib.OK              # detach
  too_big = batched.scrolling_crop_spec(31, 31, 0, pad_char=None, scroll_margins=(2, 3))
  assert lib.pcl_attach_cropper(h, C.byref(too_big), 0x20000, 0x30000) == _lib.ERR_INVALID
  drape = batched.scrolling_crop_spec(5, 5, 0, pad_char=' ', scroll_margins=(None, None),
                                      track=[-1, 1])
  assert lib.pcl_attach_cropper(h, C.byref(drape), 0x20000, 0x30000) == _lib.ERR_UNSUPPORTED
  no_such = batched.scrolling_crop_spec(5, 5, 0, pad_char=' ', scroll_margins=(None, None),
                                        track=[9])
  assert lib.pcl_attach_cropper(h, C.byref(no_such), 0x20000, 0x30000) == _lib.ERR_INVALID
  lib.pcl_destroy(h)

  other = lowering.lower(g_warehouse.make_game(levels.warehouse_level(1, shape=(20, 24))))
  lib, h = _bound_handle(other)
  crop = batched.scrolling_crop_spec(5, 5, 0, pad_char=' ', scroll_margins=(None, None))
  assert lib.pcl_attach_cropper(h, C.byref(crop), 0x20000, 0x30000) == _lib.ERR_UNSUPPORTED
  lib.pcl_destroy(h)


def test_crop_handoff_mode_checks_on_cpu():
  """pcl_crop_handoff refuses inconsistent hand-off descriptions before it launches:
  unknown mode bits, split phase with fewer than three buffer parts, record sizes."""
  import ctypes as C
  from pycolab_b200 import batched
  art = levels.scrolly_maze_level(3, world_shape=(33, 33), board_shape=(16, 16))
  lib, h = _bound_handle(lowering.lower(g_scrolly.make_game(*art)))
  crop = batched.scrolling_crop_spec(9, 9, 0, pad_char=' ', scroll_margins=(None, None))
  out = _lib.Outputs(0x1000, 0x2000, 0x3000, 0x4000, 0x5000)

  def call(**kw):
    x = _lib.HandoffState()
    x.n_peers, x.rank, x.record_bytes, x.rows, x.first_row = 1, 0, 96, 4, 0
    x.d_peer_base[0], x.d_peer_flags[0], x.d_local = 0x6000, 0x7000, 0x8000
    for k, v in kw.items():
      setattr(x, k, v)
    return lib.pcl_crop_handoff(h, C.byref(crop), 0x9000, 0xa000, C.byref(out), C.byref(x), None)

  assert call(mode=8) == _lib.ERR_INVALID                              # unknown bit
  assert call(mode=_lib.HANDOFF_LAG, n_bufs=2) == _lib.ERR_INVALID     # split phase needs 3 parts
  assert call(mode=_lib.HANDOFF_LAG) == _lib.ERR_INVALID               # n_bufs 0 means 2
  assert call(n_bufs=9) == _lib.ERR_INVALID
  assert call(record_bytes=90) == _lib.ERR_INVALID                     # not a multiple of 16
  assert call(record_bytes=80) == _lib.ERR_INVALID                     # too small for 81 + 9 bytes
  assert call(rows=3) == _lib.ERR_INVALID                              # this rank's rows do not fit
  assert call(rank=1) == _lib.ERR_INVALID
  lib.pcl_destroy(h)
