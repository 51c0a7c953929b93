"""Capture the known answers of the reference's `tests/engine_test.py`.

    python tests/golden/make_engine_kats.py        # build container only

`engine_test.py` states its expectations inline — `expectBoard(art)` callables
injected before an entity's update (the board THAT entity must see: the staged
renders between update groups, engine.py:725-735), `assertBoard(observation.board,
art)` on what `play()` returns, plain asserts on reward / discount — and drives
Plot directives (`add_reward`, `terminate_episode`, `change_z_order`) from injected
callables.  This script runs the unmodified test module with those helpers
wrapped and records, per engine and frame: the action, the hand-drawn art each
entity was promised and the art asserted on the returned observation, the Plot
directive calls made during the frame, and what the reference returned (board,
reward, discount, game_over, z-order, every layer).  It also records every call
of the observation post-processors (`rendering.Observation*`): arguments, input
board and output array.  Output: `tests/golden/reference_engine_kats.json`,
replayed on the oracle by tests/test_reference_engine_kats.py.

Shims for this image (the reference source is untouched): `EngineTest._assertMask`
parses its '0'/'1' art with `.astype(bool)`, which NumPy 2 turns into all-True; it
is replaced by the comparison it meant (`art == '1'`).
"""

import json
import os
import sys
import unittest

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import refdriver

refdriver._import()
from pycolab import ascii_art
from pycolab import rendering
from pycolab import things as plab_things
from pycolab.prefab_parts import drapes as prefab_drapes
from pycolab.prefab_parts import sprites as prefab_sprites
from pycolab.tests import engine_test
from pycolab.tests import test_things as tt

from make_kats import art_of, bits_of, plain, update_groups

ENGINES = {}          # id(engine) -> record
ORDER = []            # records in creation order
OBSERVERS = []        # post-processor calls
CURRENT = [None]      # test id
NESTED = [0]          # depth of post-processor calls


def snapshot(engine):
  snap = dict(rows=engine.rows, cols=engine.cols, frame=engine.the_plot.frame,
              backdrop=art_of(engine.backdrop.curtain), z_order=list(engine.z_order),
              groups=[[e.character for e in ents] for _, ents in update_groups(engine)],
              walkers={}, sprites={}, drapes={})
  for ch, thing in engine.things.items():
    if isinstance(thing, prefab_sprites.MazeWalker):
      snap['walkers'][ch] = dict(
          position=list(thing.position), virtual_position=list(thing.virtual_position),
          visible=bool(thing.visible), prior_visible=None,
          impassable=''.join(sorted(thing.impassable)), confined=bool(thing._confined_to_board),
          egocentric=bool(thing._egocentric_scroller), group=thing._scrolling_group)
    elif isinstance(thing, plab_things.Sprite):
      snap['sprites'][ch] = dict(position=list(thing.position), visible=bool(thing.visible))
    elif isinstance(thing, prefab_drapes.Scrolly):
      return None
    else:
      snap['drapes'][ch] = bits_of(thing.curtain)
  return snap


def register(engine, occlusion):
  rec = dict(test=CURRENT[0], occlusion_in_layers=bool(occlusion), snapshot=None, frames=[],
             pending={}, directives=[], last_board=None)
  ENGINES[id(engine)] = rec
  ORDER.append(rec)
  plot = engine.the_plot
  for name in ('add_reward', 'terminate_episode', 'change_z_order', 'change_default_discount'):
    real = getattr(plot, name)

    def logged(*args, _name=name, _real=real, **kwargs):
      rec['directives'].append([_name, plain(list(args)), plain(kwargs)])
      return _real(*args, **kwargs)
    setattr(plot, name, logged)
  real_showtime, real_play = engine.its_showtime, engine.play

  def frame(action, call):
    if rec.get('inside'):                 # its_showtime() is play(None) inside (engine.py:581)
      return call()
    rec['inside'] = True
    try:
      return record(action, call)
    finally:
      rec['inside'] = False

  def record(action, call):
    if rec['snapshot'] is None:
      rec['snapshot'] = snapshot(engine) or 'unsupported'
    rec['directives'] = []
    expected, rec['pending'] = rec['pending'], {}
    observation, reward, discount = call()
    rec['last_board'] = observation.board
    rec['frames'].append(dict(
        action=plain(action), expect_seen=expected, expect_final=None,
        directives=rec['directives'], board=art_of(observation.board), reward=plain(reward),
        discount=plain(discount), game_over=bool(engine.game_over),
        z_order=list(engine.z_order),
        layers={ch: bits_of(mask) for ch, mask in observation.layers.items()}))
    return observation, reward, discount

  engine.its_showtime = lambda: frame(None, real_showtime)
  engine.play = lambda actions: frame(actions, lambda: real_play(actions))


def install():
  real_make = ascii_art.ascii_art_to_game

  def make(*args, **kwargs):
    engine = real_make(*args, **kwargs)
    register(engine, kwargs.get('occlusion_in_layers', True))
    return engine
  engine_test.ascii_art.ascii_art_to_game = make

  real_expect = tt.PycolabTestCase.expectBoard

  def expect_board(self, art, err_msg=''):
    fn = real_expect(self, art, err_msg)
    fn.kat_art = list(art)
    return fn
  tt.PycolabTestCase.expectBoard = expect_board

  real_pre = tt.pre_update

  def pre_update(engine, character, thing_to_do):
    rec = ENGINES.get(id(engine))
    if rec is not None and hasattr(thing_to_do, 'kat_art'):
      rec['pending'][character] = thing_to_do.kat_art
    return real_pre(engine, character, thing_to_do)
  tt.pre_update = pre_update
  engine_test.tt.pre_update = pre_update

  real_assert = tt.PycolabTestCase.assertBoard

  def assert_board(self, actual_board, art, err_msg=''):
    for rec in ORDER:
      # (expectBoard callables assert on the same array object from inside update():
      # only an assertion made BETWEEN frames is about the returned observation)
      if rec['last_board'] is actual_board and rec['frames'] and not rec.get('inside'):
        rec['frames'][-1]['expect_final'] = list(art)
    return real_assert(self, actual_board, art, err_msg)
  tt.PycolabTestCase.assertBoard = assert_board

  def assert_mask(self, actual_mask, mask_art, err_msg=''):   # NumPy-2 shim, see docstring
    want = np.array([[c == '1' for c in row] for row in mask_art], dtype=bool)
    np.testing.assert_array_equal(np.asarray(actual_mask).astype(bool), want, err_msg)
  engine_test.EngineTest._assertMask = assert_mask

  for kind in ('ObservationCharacterRepainter', 'ObservationToArray', 'ObservationToFeatureArray'):
    cls = getattr(rendering, kind)
    real_init, real_call = cls.__init__, cls.__call__

    def init(self, *args, _real=real_init, **kwargs):
      self._kat_args, self._kat_kwargs = args, kwargs
      _real(self, *args, **kwargs)

    def call(self, observation, _real=real_call, _kind=kind):
      NESTED[0] += 1                      # a repainter runs a to-array converter inside
      try:
        out = _real(self, observation)
      finally:
        NESTED[0] -= 1
      if NESTED[0]:
        return out
      result = out.board if hasattr(out, 'board') else out
      kwargs = dict(self._kat_kwargs)
      if 'dtype' in kwargs and kwargs['dtype'] is not None:
        kwargs['dtype'] = np.dtype(kwargs['dtype']).name
      OBSERVERS.append(dict(
          test=CURRENT[0], kind=_kind, args=plain(list(self._kat_args)), kwargs=plain(kwargs),
          board=art_of(observation.board), out=np.asarray(result).tolist(),
          out_dtype=np.asarray(result).dtype.name, out_shape=list(np.asarray(result).shape)))
      return out
    cls.__init__, cls.__call__ = init, call


class Tracker(unittest.TextTestResult):
  def startTest(self, test):
    CURRENT[0] = test.id().split('.', 2)[-1]
    super(Tracker, self).startTest(test)


def main():
  assert refdriver.available(), refdriver.MISSING
  install()
  suite = unittest.defaultTestLoader.loadTestsFromModule(engine_test)
  result = unittest.TextTestRunner(verbosity=1, resultclass=Tracker).run(suite)
  assert result.wasSuccessful(), 'the reference failed its own tests'
  engines = []
  for rec in ORDER:
    if rec['snapshot'] in (None, 'unsupported') or not rec['frames']:
      continue
    engines.append(dict(test=rec['test'], occlusion_in_layers=rec['occlusion_in_layers'],
                        snapshot=rec['snapshot'], frames=rec['frames']))
  path = os.path.join(HERE, 'reference_engine_kats.json')
  with open(path, 'w') as f:
    json.dump(plain(dict(engines=engines, observers=OBSERVERS)), f, separators=(',', ':'),
              default=lambda o: o.item())
  print('%d engines (%d frames, %d promised boards, %d asserted observations), %d observer '
        'calls -> %s (%.1f KiB)' % (
            len(engines), sum(len(e['frames']) for e in engines),
            sum(len(fr['expect_seen']) for e in engines for fr in e['frames']),
            sum(fr['expect_final'] is not None for e in engines for fr in e['frames']),
            len(OBSERVERS), path, os.path.getsize(path) / 1024.0))
  for e in engines:
    print('  %-58s %2d frames' % (e['test'], len(e['frames'])))


if __name__ == '__main__':
  main()
