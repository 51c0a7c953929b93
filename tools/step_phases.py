#!/usr/bin/env python
"""Where one scrolly_maze_step launch spends its time, from stamps inside the kernel.

    python tools/step_phases.py --out DIR            # build the stamped library, run, print
    python tools/step_phases.py --out DIR --build-only
    python tools/step_phases.py --out DIR --lib DIR/libpcl.so

The stamped build (-DPCL_STEP_PHASES, scrolly_maze.cu) has lane 0 of every warp
record %globaltimer and clock64() at seven points of the step, plus %smid.  The
library is compiled into DIR (the tree's own build is not touched) and loaded
through PCL_LIB_PATH.  The workload is bench.py's headline: 4096 envs x 6
rotating batches, the same generated levels and actions, K steps replayed as one
CUDA graph; the stamps of the last launch are read back.

Printed per phase: median and p95 across warps of the time since the previous
stamp (SM cycles, and ns at the measured clock), the share of the median warp's
entry-to-paint-end span, and the spread across SMs of the earliest start of each
phase (globaltimer), which shows whether the wave's warps move in lock-step.
The stamps perturb absolute times: read them for shares and ordering only.
"""

import argparse
import concurrent.futures
import ctypes
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'pycolab_b200', 'csrc')
PHASES = ['entry', 'griddepcontrol.wait', 'records landed', 'second batch issued',
          'cp.async drained', 'paint start', 'paint end']
K_PHASES, K_ENVS, K_WORDS = 7, 8192, 16        # scrolly_maze.cu kPhases / kPhaseEnvs / kPhaseWords


def build(out):
  """nvcc every source of the Makefile with -DPCL_STEP_PHASES into out/libpcl.so."""
  mk = open(os.path.join(CSRC, 'Makefile')).read()
  srcs = re.search(r'^SRCS := (.*)$', mk, re.M).group(1).split()
  nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
  arch = ['-gencode', 'arch=compute_100a,code=sm_100a']
  flags = arch + ['-O3', '-std=c++17', '-lineinfo', '--use_fast_math', '-Xcompiler', '-fPIC',
                  '-cudart', 'static', '-DPCL_STEP_PHASES']
  os.makedirs(out, exist_ok=True)

  def one(src):
    obj = os.path.join(out, src[:-3] + '.o')
    subprocess.check_call([nvcc] + flags + ['-c', os.path.join(CSRC, src), '-o', obj])
    return obj

  with concurrent.futures.ThreadPoolExecutor(8) as ex:
    objs = list(ex.map(one, srcs))
  lib = os.path.join(out, 'libpcl.so')
  subprocess.check_call([nvcc] + arch + ['-shared', '-cudart', 'static', '-o', lib] + objs +
                        ['-ldl'])
  for o in objs:
    os.remove(o)
  return lib


def run(lib, steps, warmup):
  os.environ['PCL_LIB_PATH'] = os.path.abspath(lib)
  sys.path.insert(0, ROOT)
  import torch
  import bench
  from pycolab_b200 import batched, lowering
  from pycolab_b200.games import scrolly_maze

  dev = torch.device('cuda', 0)
  torch.cuda.set_device(dev)
  B, R = bench.BATCH_PER_GPU, bench.ROTATION
  arts = bench.make_levels(bench.N_LEVELS)
  lowered = [lowering.lower(scrolly_maze.make_game(*a)) for a in arts]
  engines = [batched.BatchedEngine(lowered, batch=B, device=0, env_offset=r * B)
             for r in range(R)]
  for e in engines:
    e.its_showtime()
  rs = np.random.RandomState(1234)
  actions = torch.from_numpy(rs.randint(0, bench.ACTIONS, size=(warmup + steps, B))
                             .astype(np.int32)).to(dev)
  timed = bench.Timed(torch, dev, lambda t: engines[t % R].play(actions[t]), warmup, steps)
  timed.warm()
  ms = timed.time_ms(torch.cuda.synchronize) / steps
  torch.cuda.synchronize()
  errors = max(int(e.error_codes().abs().max()) for e in engines)

  c = ctypes.CDLL(os.environ['PCL_LIB_PATH'])
  buf = np.zeros((K_ENVS, K_WORDS), dtype=np.uint64)
  rc = c.pcl_step_phases_read(buf.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(buf.nbytes))
  assert rc == 0, 'pcl_step_phases_read: cuda error %d' % rc
  buf = buf[:B].astype(np.int64)
  gt, clk, sm = buf[:, :K_PHASES], buf[:, K_PHASES:2 * K_PHASES], buf[:, 2 * K_PHASES]
  # warps that reached the end of the paint loop this launch (skip an epilogue-less exit)
  ok = (gt[:, -1] >= gt[:, 0]) & (gt[:, 0] > 0)
  gt, clk, sm = gt[ok], clk[ok], sm[ok]
  span_ns = gt[:, -1] - gt[:, 0]
  span_clk = clk[:, -1] - clk[:, 0]
  mhz = float(np.median(span_clk / np.maximum(span_ns, 1))) * 1e3
  lines = ['# scrolly_maze_step phase stamps, last launch of %d (graph replay), %d warps, '
           '%.4f ms/step with stamps, env_errors %d, %d SMs, clock %.0f MHz (clock64 / globaltimer)'
           % (steps, len(gt), ms, errors, len(np.unique(sm)), mhz)]
  lines.append('# %-22s %10s %10s %8s %8s %7s %16s' % (
      'phase (since previous)', 'med cyc', 'p95 cyc', 'med ns', 'p95 ns', 'share',
      'SM start spread'))
  total = float(np.median(span_clk))
  t0 = gt[:, 0].min()
  for i in range(K_PHASES):
    d = clk[:, i] - clk[:, i - 1] if i else np.zeros(len(clk), np.int64)
    # per SM: earliest stamp i, then the spread of that across SMs (ns after the first entry)
    first = np.array([gt[sm == s, i].min() for s in np.unique(sm)]) - t0
    spread = '%d..%d ns' % (first.min(), first.max())
    lines.append('  %-22s %10.0f %10.0f %8.0f %8.0f %6.1f%% %16s' % (
        PHASES[i], np.median(d), np.percentile(d, 95), np.median(d) / mhz * 1e3,
        np.percentile(d, 95) / mhz * 1e3, 100.0 * np.median(d) / total if total else 0.0, spread))
  lines.append('  %-22s %10.0f %10.0f %8.0f %8.0f' % (
      'entry -> paint end', total, np.percentile(span_clk, 95), np.median(span_ns),
      np.percentile(span_ns, 95)))
  lines.append('  first entry -> last paint end across the grid: %d ns' % (gt[:, -1].max() - t0))
  return '\n'.join(lines)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', required=True, help='directory for the stamped library')
  ap.add_argument('--lib', help='use this stamped libpcl.so instead of building one')
  ap.add_argument('--build-only', action='store_true')
  ap.add_argument('--steps', type=int, default=600)
  ap.add_argument('--warmup', type=int, default=30)
  args = ap.parse_args()
  lib = args.lib or build(args.out)
  if args.build_only:
    print(lib)
    return
  print(run(lib, args.steps, args.warmup))


if __name__ == '__main__':
  main()
