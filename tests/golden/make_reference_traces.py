"""Record the original pycolab's traces of the scenarios in tests/reference_trace.py.

    PYCOLAB_UPSTREAM=<dir holding the upstream pycolab package> \\
        python tests/golden/make_reference_traces.py

Writes `tests/golden/reference_traces.npz` (one uint32 array per scenario: the
chained CRC checkpoints, the final CRC and the record count), replayed on the
oracle by tests/test_oracle_vs_reference.py, and
`tests/golden/reference_observers.npz`, the original's observation
post-processors on a few warehouse boards (tests/test_observers.py), and
`tests/golden/reference_lowerings.json`, a digest of how each of the original's
example files (and one game of its test fixtures) lowers when loaded through
`compat` (tests/test_host.py and the per-game tests).  The oracle side builds its
games from art this repository holds (the stock-level goldens, the package's
GAME_ART / LEVELS); this script checks that art is the original's before it
records anything.
"""

import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import refdriver

assert refdriver.available(), refdriver.MISSING
import golden_cases as gc
import reference_trace as rt


def check_stock_art():
  """The art OracleSide uses is the original's."""
  for level in (0, 1, 2):
    assert gc.scrolly_art(gc.load('scrolly_stock_L%d' % level)) == \
        tuple(refdriver.ref_stock_scrolly_art(level))
    art, wlb = refdriver.ref_stock_warehouse_art(level)
    assert gc.warehouse_art(gc.load('warehouse_stock_L%d' % level)) == (art, wlb)
    want = [bytes(r).decode('ascii') for r in gc.load('aperture_stock_L%d' % level)['art']]
    assert want == refdriver.ref_aperture_art(level)
  from pycolab_b200 import levels
  from pycolab_b200.games import apprehend, fluvial_natation, shockwave
  assert levels.marauders_level() == refdriver.ref_stock_marauders_art()
  for kind in rt.games.CLASSIC_KINDS:
    ours = importlib.import_module('pycolab_b200.games.classics.' + kind).GAME_ART
    assert list(ours) == refdriver.ref_classic_art(kind), kind
  assert list(fluvial_natation.GAME_ART) == refdriver.ref_fluvial_art()
  from pycolab.examples import apprehend as ref_apprehend
  from pycolab.examples import shockwave as ref_shockwave
  assert list(apprehend.GAME_ART) == list(ref_apprehend.GAME_ART)
  assert list(shockwave.LEVELS[0]) == list(ref_shockwave.LEVELS[0])


def main():
  check_stock_art()
  side = refdriver.ReferenceSide()
  out = {}
  for key, (scenario, args) in sorted(rt.cases().items()):
    trace, facts = scenario(side, *args)
    out[key] = trace.result()
    print(key, trace.records, 'records', facts)
  save('reference_traces.npz', out)
  lowerings = {key: rt.lowering_digest(game) for key, game in upstream_lowerings()}
  path = os.path.join(HERE, 'reference_lowerings.json')
  with open(path, 'w') as f:
    json.dump(lowerings, f, indent=1, sort_keys=True)
    f.write('\n')
  print('wrote', path, len(lowerings), 'lowerings')
  from pycolab import rendering
  import test_observers
  save('reference_observers.npz', test_observers.observer_outputs(
      rendering, test_observers._boards('warehouse_stock_L1')))


def upstream_lowerings():
  """(key, lowered game) of the original's example files and test fixtures,
  loaded unmodified through `compat` (its `pycolab` is this package)."""
  import random
  from pycolab_b200 import compat, lowering
  saved = {k: v for k, v in sys.modules.items() if k == 'pycolab' or k.startswith('pycolab.')}
  compat.uninstall()
  compat.install()
  base = os.path.join(refdriver.REFERENCE_ROOT, 'pycolab')
  load = lambda name: compat.load_example(os.path.join(base, name + '.py'))
  try:
    out = []
    m = load('examples/scrolly_maze')
    out += [('scrolly_maze_%d' % l, m.make_game(l)) for l in (0, 1, 2)]
    m = load('examples/warehouse_manager')
    out += [('warehouse_manager_%d' % l, m.make_game(l)) for l in (0, 1, 2)]
    out.append(('extraterrestrial_marauders', load('examples/extraterrestrial_marauders').make_game()))
    m = load('examples/better_scrolly_maze')
    out += [('better_scrolly_maze_%d' % l, m.make_game(l)) for l in (0, 1, 2)]
    for kind in rt.games.CLASSIC_KINDS:
      out.append((kind, load('examples/classics/' + kind).make_game()))
    m = load('examples/aperture')
    out += [('aperture_%d' % l, m.make_game(l)) for l in (0, 1, 2)]
    out.append(('fluvial_natation', load('examples/fluvial_natation').make_game()))
    random.seed(11)
    out.append(('apprehend', load('examples/apprehend').make_game()))
    with rt.sorted_default_schedule():
      out.append(('hello_world', load('examples/hello_world').make_game()))
    out.append(('shockwave', load('examples/shockwave').make_game(0)))
    m = load('examples/ordeal')
    aa = m.ascii_art          # the original builds its chapters inside make_game() (ordeal.py:77-93)
    out.append(('ordeal_castle', aa.ascii_art_to_game(
        m.GAME_ART_CASTLE, what_lies_beneath=' ', sprites=dict(P=m.PlayerSprite, D=m.DragonduckSprite),
        update_schedule=['P', 'D'], z_order=['D', 'P'])))
    out.append(('ordeal_cavern', aa.ascii_art_to_game(
        m.GAME_ART_CAVERN, what_lies_beneath=' ', sprites=dict(P=m.PlayerSprite),
        drapes=dict(S=m.SwordDrape), update_schedule=['P', 'S'])))
    out.append(('ordeal_kansas', aa.ascii_art_to_game(
        m.GAME_ART_KANSAS, what_lies_beneath='~', sprites=dict(P=m.PlayerSprite))))
    tt = load('tests/test_things')
    kw, _ = gc.fixture_kwargs(gc.load('fixture_scrolly_0'))
    aa = sys.modules['pycolab.ascii_art']
    shape = (len(kw['art']), len(kw['art'][0]))
    sprites = {ch: aa.Partial(tt.TestMazeWalker, impassable=w.get('impassable', ''),
                              confined_to_board=w.get('confined', False),
                              egocentric_scroller=w.get('egocentric', False))
               for ch, w in kw['walkers'].items()}
    drapes = {ch: aa.Partial(tt.TestScrolly, board_shape=shape, whole_pattern=sc['pattern'],
                             board_northwest_corner=sc['corner'], scroll_margins=sc['margins'])
              for ch, sc in kw['scrollys'].items()}
    out.append(('test_things_fixture_scrolly_0', aa.ascii_art_to_game(
        kw['art'], ' ', sprites, drapes, update_schedule=kw['update_schedule'],
        z_order=kw['z_order'])))
    return [(key, lowering.lower(game)) for key, game in out]
  finally:
    compat.uninstall()
    sys.modules.update(saved)


def save(name, arrays):
  path = os.path.join(HERE, name)
  np.savez_compressed(path, **arrays)
  print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
  main()
