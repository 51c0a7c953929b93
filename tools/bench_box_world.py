#!/usr/bin/env python
"""Box-World step throughput on one GPU: the box_world program over a pool of
generated levels, level rotation on, random moves drawn on the device.

For each batch size, K steps are captured as ONE CUDA graph (one `pcl_run` call of
K `pcl_step` launches through the C ABI), replayed once to warm up, then timed with
CUDA events over --reps replays.  Prints one JSON line (and writes it to --out):
µs per step, env-steps/s and the bytes a running step moves per env, computed from
the shapes, with the GPU's name, power limit and max SM clock read in the same run.

The working set is about 1 KB per env (records, the cell plane, the board), so at
these batch sizes it lives in the 126 MB L2.  That is how the engine is used: the
same envs are stepped again and again.  The numbers are L2-resident on purpose.

    python tools/bench_box_world.py --pool 16384 --steps 200 --out /tmp/bench_box_world.json
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DEFAULT = (12, (1, 2, 3, 4), (0, 1, 2, 3, 4), (0,), 1)


def gpu_info(index):
  q = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm',
                      '--format=csv,noheader'], capture_output=True, text=True)
  name, power, clock = [f.strip() for f in q.stdout.strip().split(',')]
  return {'gpu': name, 'power_limit': power, 'max_sm_clock': clock}


def build_pool(n):
  from pycolab_b200 import lowering
  from pycolab_b200.games import box_world
  return [lowering.lower(box_world.make_game(*DEFAULT, random_state=np.random.RandomState(s)))
          for s in range(n)]


def bytes_per_env_step(game):
  """DRAM/L2 traffic of one running step of one env, from the shapes: reads of the
  sprite record (32 B), four plot words, the action and the live plane; writes of the
  board, the records, the four outputs and at most two plane bytes."""
  plane = game.rows * game.pitch
  reads = 32 + 16 + 4 + plane
  writes = plane + 32 + 16 + (4 + 1 + 4 + 1) + 2
  return reads + writes


def time_engine(torch, eng, steps, reps):
  B = eng.batch
  gen = torch.Generator(device=eng.device)
  gen.manual_seed(0)
  actions = torch.randint(0, 4, (steps, B), device=eng.device, dtype=torch.int32, generator=gen)
  eng.its_showtime()
  eng.run(actions)                       # warm: module load, first restarts
  torch.cuda.synchronize()
  graph = torch.cuda.CUDAGraph()
  stream = torch.cuda.Stream()
  with torch.cuda.stream(stream):
    with torch.cuda.graph(graph, stream=stream):
      eng.run(actions)
  graph.replay()
  torch.cuda.synchronize()
  times = []
  for _ in range(reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    graph.replay()
    b.record()
    b.synchronize()
    times.append(a.elapsed_time(b) * 1e3 / steps)
  assert not eng.error_codes().any()
  return float(np.median(times)), float(np.min(times)), float(np.max(times))


def main():
  ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
  ap.add_argument('--pool', type=int, default=16384)
  ap.add_argument('--batches', default='4096,16384,65536')
  ap.add_argument('--steps', type=int, default=200)
  ap.add_argument('--reps', type=int, default=20)
  ap.add_argument('--out', default=None)
  args = ap.parse_args()
  import torch
  from pycolab_b200 import batched
  if not torch.cuda.is_available():
    raise SystemExit('bench_box_world needs a CUDA device')
  info = gpu_info(torch.cuda.current_device())
  t0 = time.time()
  pool = build_pool(args.pool)
  pool_s = time.time() - t0
  per_env = bytes_per_env_step(pool[0])
  rows = []
  runs = [(int(b), True) for b in args.batches.split(',')] + [(4096, False)]
  for B, cycle in runs:
    eng = batched.BatchedEngine(pool, batch=B, cycle_levels=cycle)
    med, lo, hi = time_engine(torch, eng, args.steps, args.reps)
    rows.append({'batch': B, 'cycle_levels': cycle, 'us_per_step': round(med, 3),
                 'us_min': round(lo, 3), 'us_max': round(hi, 3),
                 'env_steps_per_s': round(B / med * 1e6),
                 'bytes_per_env_step': per_env,
                 'achieved_GB_per_s': round(B * per_env / med * 1e-3, 1)})
    eng.close()
    del eng
    torch.cuda.empty_cache()
  result = dict(info, program='box_world', board='%dx%d' % (pool[0].rows, pool[0].cols),
                pool_levels=args.pool, pool_build_s=round(pool_s, 1), steps_per_graph=args.steps,
                reps=args.reps, actions='uniform 0..3 drawn on the device', l2_resident=True,
                results=rows)
  line = json.dumps(result)
  print(line)
  if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
      f.write(line + '\n')


if __name__ == '__main__':
  main()
