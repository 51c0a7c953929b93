"""ctypes binding of libpcl.so (include/pcl.h).

The product path has no CPU fallback: if the CUDA library is missing or fails
to load, everything that would step an environment raises `PclLibraryError`.
"""

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PCL_LIB_PATH: development switch for A/B runs of two builds in one process series.
LIB_PATH = os.environ.get('PCL_LIB_PATH') or os.path.join(_HERE, 'libpcl.so')

ABI_VERSION = 2
MAX_SPRITES = 16
MAX_DRAPES = 8
MAX_TRACK = 4                # entities one ScrollingCropper can follow (pcl_crop_spec.track)
SPRITE_WORDS = 8
DRAPE_WORDS = 8
PLOT_WORDS = 16
MT_WORDS = 625
MAX_SCROLL_GROUPS = 4
GROUP_WORDS = 4
G_ORDER_R, G_ORDER_C, G_ORDER_FRAME, G_EGO_MASK = range(4)
FIXTURE_DIRECTIVES = 4       # (opcode, argument) pairs per PROG_FIXTURE action row
DIR_NONE, DIR_ADD_REWARD, DIR_TERMINATE, DIR_DEFAULT_DISCOUNT, DIR_Z_ORDER = range(5)
HOST_SLOTS = 8               # pcl_step_host_async completion slots
NEVER = -(2 ** 31)           # INT32_MIN: "-inf"/None frame
ACTION_NONE = -1

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_UNBOUND, ERR_NOMEM = 0, -1, -2, -3, -4, -5

ENV_ERR_ORDER_MISMATCH = 0x1
ENV_ERR_SECOND_ORDER = 0x2
ENV_ERR_EMPTY_CHOICE = 0x4
ENV_ERR_INDEX = 0x8
ENV_ERR_BAD_Z = 0x10

PROG_NONE, PROG_SCROLLY_MAZE, PROG_WAREHOUSE, PROG_MARAUDERS, PROG_FIXTURE = 0, 1, 2, 3, 4
PROG_BETTER_SCROLLY, PROG_CLASSICS, PROG_APERTURE, PROG_ORDEAL, PROG_HELLO = 5, 6, 7, 8, 9
PROG_APPREHEND, PROG_SHOCKWAVE, PROG_BOX_WORLD = 10, 11, 12
ORDEAL_NEXT_UNSET, ORDEAL_NEXT_NONE, ORDEAL_CASTLE, ORDEAL_CAVERN, ORDEAL_KANSAS = -1, 0, 1, 2, 3
CLASSIC_FOUR_ROOMS, CLASSIC_CLIFF_WALK, CLASSIC_CHAIN_WALK, CLASSIC_FLUVIAL = 0, 1, 2, 3

# Record word indices (pcl.h enums).
S_ROW, S_COL, S_VROW, S_VCOL, S_FLAGS, S_AUX0, S_AUX1, S_AUX2 = range(8)
D_CORNER_R, D_CORNER_C, D_PRE_R, D_PRE_C, D_LAST_FRAME, D_AUX0, D_AUX1, D_AUX2 = range(8)
(P_FRAME, P_GAME_OVER, P_ERROR, P_EPISODES, P_ORDER_R, P_ORDER_C, P_ORDER_FRAME,
 P_EGO_MASK, P_AUX0, P_AUX1, P_AUX2, P_AUX3, P_CROP_R, P_CROP_C, P_CROP_INIT,
 P_RESERVED) = range(16)


class PclLibraryError(RuntimeError):
  """libpcl.so is missing / not loadable: there is no CPU path to fall back to."""


class PclError(RuntimeError):
  """A libpcl entry point returned a negative status."""

  def __init__(self, status, what):
    self.status = status
    RuntimeError.__init__(self, '%s failed: %s (%d)' % (what, status_string(status), status))


_N = MAX_SPRITES + MAX_DRAPES


class Spec(C.Structure):
  _fields_ = [
      ('abi_version', C.c_int32), ('program', C.c_int32),
      ('rows', C.c_int32), ('cols', C.c_int32), ('pitch', C.c_int32),
      ('n_sprites', C.c_int32), ('n_drapes', C.c_int32), ('auto_reset', C.c_int32),
      ('pattern_rows', C.c_int32), ('pattern_cols', C.c_int32),
      ('pattern_words', C.c_int32), ('bits_words', C.c_int32),
      ('sprite_char', C.c_uint8 * MAX_SPRITES), ('drape_char', C.c_uint8 * MAX_DRAPES),
      ('impassable', (C.c_uint32 * 4) * MAX_SPRITES),
      ('sprite_confined', C.c_int32 * MAX_SPRITES),
      ('sprite_egocentric', C.c_int32 * MAX_SPRITES),
      ('margins', (C.c_int32 * 2) * MAX_DRAPES),
      ('z_order', C.c_uint8 * _N),
      ('n_groups', C.c_int32),
      ('group_len', C.c_int32 * _N),
      ('group_chars', C.c_uint8 * _N),
      ('drape_kind', C.c_int32 * MAX_DRAPES),
      ('program_arg', C.c_int32 * 8),
      ('n_scroll_groups', C.c_int32),
      ('sprite_group', C.c_int32 * MAX_SPRITES),
      ('drape_group', C.c_int32 * MAX_DRAPES),
  ]


class State(C.Structure):
  _fields_ = [
      ('d_backdrop', C.c_void_p), ('backdrop_bstride', C.c_int64),
      ('d_pattern', C.c_void_p * MAX_DRAPES), ('pattern_bstride', C.c_int64 * MAX_DRAPES),
      ('d_pattern_init', C.c_void_p * MAX_DRAPES),
      ('pattern_init_bstride', C.c_int64 * MAX_DRAPES),
      ('d_bits', C.c_void_p * MAX_DRAPES), ('bits_bstride', C.c_int64 * MAX_DRAPES),
      ('d_bits_init', C.c_void_p * MAX_DRAPES), ('bits_init_bstride', C.c_int64 * MAX_DRAPES),
      ('d_sprites', C.c_void_p), ('d_sprites_init', C.c_void_p),
      ('sprites_init_bstride', C.c_int64),
      ('d_drapes', C.c_void_p), ('d_drapes_init', C.c_void_p),
      ('drapes_init_bstride', C.c_int64),
      ('d_plot', C.c_void_p), ('d_plot_init', C.c_void_p), ('plot_init_bstride', C.c_int64),
      ('d_rng', C.c_void_p),
      ('d_z_order', C.c_void_p), ('d_z_order_init', C.c_void_p),
      ('z_order_init_bstride', C.c_int64),
      ('d_groups', C.c_void_p), ('d_groups_init', C.c_void_p),
      ('groups_init_bstride', C.c_int64),
      ('d_level', C.c_void_p),
  ]


class Outputs(C.Structure):
  _fields_ = [('d_board', C.c_void_p), ('d_reward', C.c_void_p),
              ('d_has_reward', C.c_void_p), ('d_discount', C.c_void_p),
              ('d_done', C.c_void_p)]


class CropSpec(C.Structure):
  _fields_ = [('rows', C.c_int32), ('cols', C.c_int32), ('sprite_index', C.c_int32),
              ('pad_char', C.c_int32), ('margin_rows', C.c_int32),
              ('margin_cols', C.c_int32), ('offset_rows', C.c_int32),
              ('offset_cols', C.c_int32), ('saccade', C.c_int32),
              ('track', C.c_int32 * 4)]      # MAX_TRACK priority list, 0-terminated


MAX_PEERS = 8


HANDOFF_LAG, HANDOFF_SIGNAL_KERNEL = 1, 2


class HandoffState(C.Structure):
  """include/pcl.h pcl_handoff."""
  _fields_ = [('n_peers', C.c_int32), ('rank', C.c_int32), ('record_bytes', C.c_int32),
              ('rows', C.c_int64), ('first_row', C.c_int64),
              ('d_peer_base', C.c_void_p * MAX_PEERS), ('d_peer_flags', C.c_void_p * MAX_PEERS),
              ('d_multicast', C.c_void_p), ('d_local', C.c_void_p),
              ('n_bufs', C.c_int32), ('mode', C.c_int32)]


class ObserveSpec(C.Structure):
  _fields_ = [('depth', C.c_int32), ('dtype', C.c_int32), ('stride_b', C.c_int64),
              ('stride_d', C.c_int64), ('stride_r', C.c_int64), ('stride_c', C.c_int64)]


# name -> (restype, argtypes); every symbol include/pcl.h declares.
SYMBOLS = {
    'pcl_abi_version': (C.c_int, []),
    'pcl_struct_sizes': (C.c_int, [C.POINTER(C.c_int32)]),
    'pcl_status_string': (C.c_char_p, [C.c_int]),
    'pcl_create': (C.c_int, [C.POINTER(Spec), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'pcl_destroy': (C.c_int, [C.c_void_p]),
    'pcl_bind_state': (C.c_int, [C.c_void_p, C.POINTER(State)]),
    'pcl_reset': (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Outputs), C.c_void_p]),
    'pcl_step': (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Outputs), C.c_void_p]),
    'pcl_run': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(Outputs), C.c_void_p]),
    'pcl_step_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Outputs),
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p]),
    'pcl_run_many': (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p),
                               C.POINTER(C.c_void_p), C.c_int, C.c_void_p]),
    'pcl_step_host_async': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Outputs),
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_void_p]),
    'pcl_host_wait': (C.c_int, [C.c_void_p, C.c_int]),
    'pcl_last_error': (C.c_char_p, [C.c_void_p]),
    'pcl_render': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_void_p, C.c_void_p]),
    'pcl_layers': (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'pcl_export_curtain': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'pcl_crop': (C.c_int, [C.c_void_p, C.POINTER(CropSpec), C.c_void_p, C.c_void_p,
                           C.c_void_p, C.c_void_p]),
    'pcl_attach_cropper': (C.c_int, [C.c_void_p, C.POINTER(CropSpec), C.c_void_p, C.c_void_p]),
    'pcl_crop_tracking': (C.c_int, [C.c_void_p, C.POINTER(CropSpec), C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p]),
    'pcl_pack_handoff': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(Outputs),
                                   C.c_void_p, C.c_void_p]),
    'pcl_pack_handoff_peers': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(Outputs),
                                         C.POINTER(C.c_void_p), C.c_int32, C.c_int64,
                                         C.c_void_p]),
    'pcl_crop_handoff': (C.c_int, [C.c_void_p, C.POINTER(CropSpec), C.c_void_p, C.c_void_p,
                                   C.POINTER(Outputs), C.POINTER(HandoffState), C.c_void_p]),
    'pcl_observe': (C.c_int, [C.c_void_p, C.POINTER(ObserveSpec), C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'pcl_error_codes': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    'pcl_launch_count': (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
}

_lib = None


def load():
  """Load libpcl.so (once) and type every entry point.  Raises loudly."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise PclLibraryError(
        '%s not found: build it with `python -c "import __graft_entry__ as g; '
        'g.build()"` or `make -C pycolab_b200/csrc`.  pycolab_b200 has no CPU '
        'fallback.' % LIB_PATH)
  try:
    lib = C.CDLL(LIB_PATH)
  except OSError as e:
    raise PclLibraryError('cannot load %s: %s' % (LIB_PATH, e))
  for name, (restype, argtypes) in SYMBOLS.items():
    try:
      fn = getattr(lib, name)
    except AttributeError:
      raise PclLibraryError('%s does not export %s' % (LIB_PATH, name))
    fn.restype = restype
    fn.argtypes = argtypes
  if lib.pcl_abi_version() != ABI_VERSION:
    raise PclLibraryError('ABI mismatch: library %d, binding %d' % (
        lib.pcl_abi_version(), ABI_VERSION))
  sizes = (C.c_int32 * 4)()
  lib.pcl_struct_sizes(sizes)
  mine = [C.sizeof(Spec), C.sizeof(State), C.sizeof(Outputs), C.sizeof(CropSpec)]
  if list(sizes) != mine:
    raise PclLibraryError('struct layout mismatch between include/pcl.h and _lib.py: library '
                          '%s, binding %s (pcl_spec, pcl_state, pcl_outputs, pcl_crop_spec)' % (
                              list(sizes), mine))
  _lib = lib
  return lib


def status_string(status):
  try:
    return load().pcl_status_string(status).decode()
  except PclLibraryError:
    return 'status %d' % status


def check(status, what, handle=None):
  if status != OK:
    err = PclError(status, what)
    if status == ERR_CUDA and handle is not None:
      try:
        detail = load().pcl_last_error(handle).decode()
      except Exception:                      # noqa: BLE001 - the status itself still raises
        detail = ''
      if detail:
        err.args = ('%s [%s]' % (err.args[0], detail),)
    raise err
