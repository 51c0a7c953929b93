#!/usr/bin/env python
"""bench.py — env-steps/sec of the batched step engine (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

A "step" is one pass of the hot path (Engine.play for every env = ONE fused
kernel launch through the C ABI) over one batch of synthetic random actions.
Headline workload at every N: BASELINE.json configs[1] per GPU — scrolly_maze on
seeded generated levels, 64x64 board over a 129x129 world, 4096 envs per GPU
(weak scaling; envs shard across ranks with no data-path collective).

Printed JSON (one line, rank 0): see the task contract.
  * `value`: K steps replayed as ONE captured CUDA graph of K `pcl_step` launches
    (no host code between launches), one CUDA event pair on the launch stream,
    inputs resident in HBM, rotating over 6 independent 4096-env batches so the
    working set exceeds L2.  Max over ranks; `per_rank_ms_per_step` lists all.
  * `e2e`: the same steps through the host-buffer C-ABI entry point
    (`pcl_step_host_async` + `pcl_host_wait`): pinned HOST actions in, boards +
    reward/discount/done out to pinned HOST buffers, every step, copies inside
    the timed region, two steps in flight over the rotating batches.
  * `parity_checked`: after the timed region the oracle replays a sample of the
    BENCHMARKED envs (their own levels and action streams) and the final boards,
    rewards, discounts, done flags and sprite positions must be identical.
  * `configs`: the other BASELINE.json configurations (C3 warehouse 80x80 x8192,
    C4 marauders x4096/GPU, C5 scrolly + 9x9 crop x8192/GPU) timed the same way.
  * at N > 1 `handoff_allgather` times step + crop + hand-off of every shard's
    (crop, reward, discount, done) to every rank and checks it against NCCL.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BOARD = (64, 64)
WORLD = (129, 129)
BATCH_PER_GPU = 4096
N_LEVELS = 32
ROTATION = 6                      # independent batches stepped round-robin (> L2)
ACTIONS = 5                       # 0..4, no quit (SURVEY.md §8d)
# Algorithmic bytes per env-step, reference layout (SURVEY.md §8d, C2):
#   H*W*(1 backdrop + 2 pattern windows + 2 curtains + 1 board) + 64*S + 64
A_STEP_BYTES = 64 * 64 * 6 + 64 * 4 + 64          # 24 896
# Bytes this implementation's layout moves per env-step (DESIGN.md §4; the round-1
# definition, kept for continuity): backdrop tile 4096 + board 4096 + 2 bit-packed
# 64-row windows (64 * 2 * 8 B) + records read and written (2 * 256 B).
LAYOUT_STEP_BYTES = 4096 + 4096 + 2 * 64 * 8 + 2 * 256      # 9 728
# ... of which only these reach DRAM when levels are shared (the backdrop tile and the
# wall pattern are per-LEVEL data served from L2): board store 4096 + the per-env coin
# window (64 rows x one 32-byte sector) + records.
DRAM_STEP_BYTES = 4096 + 64 * 32 + 2 * 256                  # 6 656
PARITY_ENVS = 48                  # sampled envs the oracle replays after the timed region


def make_levels(n, seed0=1000):
  from pycolab_b200 import levels
  return [levels.scrolly_maze_level(seed0 + i, world_shape=WORLD, board_shape=BOARD)
          for i in range(n)]


def usable_cores():
  """Host threads this process may really use: the affinity mask, capped by the
  cgroup CPU quota (os.cpu_count() reports the whole machine)."""
  try:
    n = len(os.sched_getaffinity(0))
  except (AttributeError, OSError):
    n = os.cpu_count() or 1
  for path in ('/sys/fs/cgroup/cpu.max',):
    try:
      quota, period = open(path).read().split()[:2]
      if quota != 'max':
        n = max(1, min(n, int(float(quota) / float(period))))
    except (OSError, ValueError):
      pass
  try:
    q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
    p = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
    if q > 0 and p > 0:
      n = max(1, min(n, q // p))
  except (OSError, ValueError):
    pass
  return n


# ------------------------------------------------------------- CPU baselines

def reference_root():
  """Directory holding the UNMODIFIED reference package, if an offline install of it
  (`pip install --target baseline/_ref`, git-ignored) sits beside this file."""
  root = os.path.join(ROOT, 'baseline', '_ref')
  if os.path.isfile(os.path.join(root, 'pycolab', 'engine.py')):
    return root
  return None


_ENV = {}


def _make_cpu_env(seed, kind):
  """One env of the C2 workload: the reference itself (kind 'reference') built
  through its own examples/scrolly_maze.make_game on the generated art, or the
  oracle port."""
  art = make_levels(1, seed0=1000 + seed % N_LEVELS)[0]
  if kind == 'reference':
    root = reference_root()
    if root not in sys.path:
      sys.path.insert(0, root)
    import warnings
    warnings.filterwarnings('ignore')
    from pycolab.examples import scrolly_maze as m     # the reference's own module
    def make():
      saved = (m.MAZES_ART, m.MAZES_WHAT_LIES_BENEATH, m.STAR_ART)
      try:       # the example reads its art from module constants: hand it ours
        m.MAZES_ART, m.MAZES_WHAT_LIES_BENEATH, m.STAR_ART = [art[0]], [art[2]], art[1]
        return m.make_game(0)
      finally:
        m.MAZES_ART, m.MAZES_WHAT_LIES_BENEATH, m.STAR_ART = saved
    return make
  from oracle import games as ogames
  return lambda: ogames.make_scrolly_maze(art[0], art[1], '+', art[2])


def _cpu_worker(args):
  """Step one CPU env (kept alive per process) for ~budget seconds."""
  seed, budget, kind = args
  key = ('env', kind)
  if key not in _ENV:
    _ENV[('make', kind)] = _make_cpu_env(seed, kind)
    _ENV[('rs', kind)] = np.random.RandomState(1234 + seed)
    _ENV[key] = _ENV[('make', kind)]()
    _ENV[key].its_showtime()
  make, rs, env = _ENV[('make', kind)], _ENV[('rs', kind)], _ENV[key]
  steps = 0
  t0 = time.perf_counter()
  while True:
    for a in rs.randint(0, ACTIONS, size=50):
      if env.game_over:
        env = make()
        env.its_showtime()
      else:
        env.play(int(a))
      steps += 1
    el = time.perf_counter() - t0
    if el >= budget:
      _ENV[key] = env
      return steps, el


def cpu_baseline(cores, budget, kind, pool=None):
  """env-steps/sec of the CPU path on `cores` host processes (whole sample)."""
  if cores == 1 or pool is None:
    results = [_cpu_worker((0, budget, kind))]
  else:
    results = pool.map(_cpu_worker, [(i, budget, kind) for i in range(cores)], chunksize=1)
  steps = sum(r[0] for r in results)
  secs = max(r[1] for r in results)
  return steps / secs, steps


def cpu_kind():
  return 'reference' if reference_root() else 'port'


def cpu_note(kind):
  if kind == 'reference':
    return ('the unmodified reference (pycolab.examples.scrolly_maze via %s), one Engine per '
            'process, fresh Engine on game-over' % os.path.relpath(reference_root(), ROOT))
  return ('oracle port (oracle/games.py, a NumPy restatement ~2.3x faster than pycolab itself): '
          'no copy of the reference package on this box')


# ------------------------------------------------------------------- clocks

class ClockSampler(object):
  """nvidia-smi clock / throttle-reason samples during the loaded window."""
  QUERY = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
           'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
           'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index):
    self.gpu = gpu_index            # one index, or a comma-separated list
    self.proc = None
    self.path = None
    self.begin = self.end = None

  def start(self):
    try:
      fd, self.path = tempfile.mkstemp(suffix='.csv')
      os.close(fd)
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.QUERY,
           '--format=csv,noheader,nounits', '-lms', '20'],
          stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
    except OSError:
      self.proc = None

  def mark_begin(self):
    self.begin = time.time()

  def mark_end(self):
    self.end = time.time()

  def stop(self):
    import datetime
    out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
    if self.proc is None:
      return out
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except subprocess.TimeoutExpired:
      self.proc.kill()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    rows = []
    for line in open(self.path):
      f = [x.strip() for x in line.split(',')]
      if len(f) < 9:
        continue
      try:
        ts = datetime.datetime.strptime(f[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
        rows.append((ts, float(f[1]), float(f[2]),
                     [n for n, v in zip(names, f[5:9]) if v.lower().startswith('active')]))
      except ValueError:
        continue
    os.unlink(self.path)
    inside = [r for r in rows if self.begin is not None and self.end is not None
              and self.begin - 0.02 <= r[0] <= self.end + 0.02]
    window = 'loaded window'
    if not inside:                      # window shorter than the sampling period
      inside = [r for r in rows if self.begin is None or r[0] >= self.begin - 0.25]
      window = 'nearest samples (loaded window shorter than the sampling period)'
    if inside:
      out.update(sm_mhz=float(np.median([r[1] for r in inside])),
                 sm_max_mhz=float(max(r[2] for r in inside)),
                 reasons=sorted({n for r in inside for n in r[3]}),
                 samples=len(inside), window=window)
    return out


def pin_to_gpu_numa_node(torch, index, world):
  """Restrict this process (and so its pinned host buffers, first touched later) to
  the CPUs of the NUMA node its GPU hangs off: eight unpinned ranks each pulling
  boards through pinned memory otherwise contend across sockets.  Falls back to an
  even split of the nodes over the local ranks when sysfs does not name the node.
  Returns a short description for the JSON line."""
  try:
    nodes = sorted(int(d[4:]) for d in os.listdir('/sys/devices/system/node')
                   if d.startswith('node') and d[4:].isdigit())
  except OSError:
    return 'no NUMA information'
  if len(nodes) < 2:
    return 'single NUMA node'
  node, how = -1, 'sysfs'
  try:
    props = torch.cuda.get_device_properties(index)
    bus = '%04x:%02x:%02x.0' % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
    node = int(open('/sys/bus/pci/devices/%s/numa_node' % bus).read())
  except (OSError, ValueError, AttributeError):
    pass
  if node < 0:
    n_local = max(world, torch.cuda.device_count())
    node, how = nodes[min(len(nodes) - 1, index * len(nodes) // max(1, n_local))], 'even split'
  try:
    cpus = set()
    for part in open('/sys/devices/system/node/node%d/cpulist' % node).read().strip().split(','):
      lo, _, hi = part.partition('-')
      cpus.update(range(int(lo), int(hi or lo) + 1))
    cpus &= set(os.sched_getaffinity(0))
    if cpus:
      os.sched_setaffinity(0, cpus)
      return 'node %d (%s), %d cpus' % (node, how, len(cpus))
  except (OSError, ValueError):
    pass
  return 'not pinned'


# ------------------------------------------------------------ reference arm

def run_reference_arm(args, rank, world):
  """The reference's CPU path for the same metric and workload, on all host
  threads this process may use: the UNMODIFIED reference when a copy travelled
  (`baseline/_ref`), else the oracle port.  Each "step" is a bounded time slice of
  the same workload on every core."""
  if rank != 0:
    return
  import multiprocessing as mp
  cores = usable_cores()
  kind = cpu_kind()
  K, W = args.steps, args.warmup
  slice_s = max(0.05, min(1.0, 45.0 / max(1, K + W)))
  t0 = time.perf_counter()
  with mp.get_context('fork').Pool(cores) as pool:
    for _ in range(max(1, W)):
      cpu_baseline(cores, slice_s, kind, pool)
    total_steps, total_secs = 0, 0.0
    for _ in range(K):
      rate, steps = cpu_baseline(cores, slice_s, kind, pool)
      total_steps += steps
      total_secs += steps / rate
  value = total_steps / total_secs
  print(json.dumps({
      'impl': 'reference', 'metric': 'env_steps_per_sec', 'value': value,
      'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': K,
      'warmup': W, 'ms_per_step': 1000.0 * total_secs / max(1, K),
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'u8', 'data': 'synthetic',
      'config': workload_config(args.gpus),
      'cpu_baseline': {'value': value, 'unit': 'env-steps/s', 'cores': cores,
                       'value_per_core': value / cores,
                       'os_cpu_count': os.cpu_count(), 'kind': kind, 'what': cpu_note(kind),
                       'sample': '%d env-steps of the same generated 64x64 levels, one env per '
                                 'host process, %d processes' % (total_steps, cores)},
      'e2e': {'value': value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'wall_s': time.perf_counter() - t0}))


# ------------------------------------------------------------ timing helpers

class Timed(object):
  """K steps as one captured CUDA graph (fallback: a host loop), timed with one
  CUDA event pair on the launch stream."""

  def __init__(self, torch, dev, step_fn, n_warm, n_steps):
    self.torch, self.dev = torch, dev
    self.step_fn, self.n_warm, self.n_steps = step_fn, n_warm, n_steps
    self.graphs = None
    self.path = 'host loop of pcl_step calls (CUDA graph capture unavailable)'
    if os.environ.get('PCL_BENCH_NO_GRAPH') == '1':   # e.g. under a profiler
      self.path = 'host loop of pcl_step calls (PCL_BENCH_NO_GRAPH=1)'
      return
    try:
      torch.cuda.synchronize(dev)
      gw, gt = (torch.cuda.CUDAGraph() if n_warm > 0 else None), torch.cuda.CUDAGraph()
      if gw is not None:
        with torch.cuda.graph(gw):
          for t in range(n_warm):
            step_fn(t)
      with torch.cuda.graph(gt):
        for t in range(n_steps):
          step_fn(n_warm + t)
      self.graphs = (gw, gt)
      self.path = 'one CUDA graph of the K step launches (captured through the C ABI)'
    except Exception as err:      # noqa: BLE001 - fall back to the host loop
      self.path += ': %s' % (str(err).splitlines()[0][:100] if str(err) else type(err).__name__)
      try:
        torch.cuda.synchronize(dev)
      except Exception:           # noqa: BLE001
        pass

  def warm(self):
    if self.graphs:
      if self.graphs[0] is not None:
        self.graphs[0].replay()
    else:
      for t in range(self.n_warm):
        self.step_fn(t)

  def run(self):
    if self.graphs:
      self.graphs[1].replay()
    else:
      for t in range(self.n_steps):
        self.step_fn(self.n_warm + t)

  def time_ms(self, barrier):
    torch = self.torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    a.record()
    self.run()
    b.record()
    barrier()
    return float(a.elapsed_time(b))


def ramp_clocks(torch, dev, timed, seconds=0.5):
  """Bring the GPU out of idle clocks (a sub-millisecond timed region is otherwise
  at the mercy of the clock ramp) by replaying the timed graph."""
  until = time.perf_counter() + seconds
  while time.perf_counter() < until:
    for _ in range(8):
      timed.run()
    torch.cuda.synchronize(dev)


def e2e_pipelined(torch, dev, engines, actions_np, n_steps, barrier, crop_spec=None,
                  crop_states=None, warm_seconds=0.3):
  """End to end through `pcl_step_host_async`: every step copies its actions from
  pinned host memory, steps, and copies its outputs back to pinned host memory;
  step t's copies overlap step t + 1's kernel (another batch); the host collects
  step t - 1 while t is in flight.  Returns seconds for n_steps."""
  R = len(engines)
  def submit(t):
    e = engines[t % R]
    e.play_host_async(actions_np[t % len(actions_np)], slot=(t // R) % 2, crop_spec=crop_spec,
                      crop_state=None if crop_states is None else crop_states[t % R])
  def collect(t):
    return engines[t % R].host_wait((t // R) % 2)
  # Warm the pinned buffers / copy streams, then keep the pipeline busy for
  # `warm_seconds`: after an idle stretch (the CPU oracle check runs just before)
  # the SM clocks and the PCIe link take tens of milliseconds to leave their idle
  # state, and a 30 ms timed window straight after it measured 3x low
  # (profiles/r02a_e2e_probe.txt has the steady-state figures).
  for t in range(2 * R):
    submit(t)
    collect(t)
  until = time.perf_counter() + warm_seconds
  t = 0
  while time.perf_counter() < until:
    submit(t)
    if t >= 1:
      collect(t - 1)
    t += 1
  if t:
    collect(t - 1)
  torch.cuda.synchronize(dev)
  barrier()
  t0 = time.perf_counter()
  for t in range(n_steps):
    submit(t)
    if t >= 1:
      collect(t - 1)
  out = collect(n_steps - 1)
  torch.cuda.synchronize(dev)
  secs = time.perf_counter() - t0
  barrier()
  return secs, out


def pcie_probe(torch, dev, barrier, mb=64, reps=8):
  """Plain pinned D2H copy bandwidth of this rank while every rank copies at once:
  the hardware ceiling of `e2e` (boards are 4 KB per env-step)."""
  src = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
  dst = torch.empty(mb << 20, dtype=torch.uint8).pin_memory()
  dst.copy_(src)
  barrier()
  t0 = time.perf_counter()
  for _ in range(reps):
    dst.copy_(src, non_blocking=True)
  torch.cuda.synchronize(dev)
  return reps * (mb << 20) / (time.perf_counter() - t0) / 1e9


def max_over_ranks(torch, dist, dev, world, x):
  if world == 1:
    return float(x), [float(x)]
  t = torch.tensor([x], device=dev, dtype=torch.float64)
  every = [torch.zeros_like(t) for _ in range(world)]
  dist.all_gather(every, t)
  vals = [float(v.item()) for v in every]
  return max(vals), vals


# ------------------------------------------------------ stand-alone renderer

def render_microbench(engines, n=60):
  """Mean device time per launch of the stand-alone renderer (`pcl_render`,
  Engine._render + BaseObservationRenderer in the reference's byte layout):
  backdrop + 2 byte curtains + sprites -> board, rotating over the R engines'
  states (working set > L2), n launches back to back between one event pair."""
  import ctypes as C
  import torch
  from pycolab_b200 import _lib
  lib = _lib.load()
  sets = []
  for eng in engines:
    B, H, pitch = eng.batch, eng.rows, eng.pitch
    dev = eng.device
    curtains = torch.zeros((B, 2, H, pitch), dtype=torch.uint8, device=dev)
    curtains[:, 0, :, :eng.cols] = eng.curtain('#')
    curtains[:, 1, :, :eng.cols] = eng.curtain('@')
    # reference layout for the stand-alone renderer: one backdrop per env
    backdrop = (eng.backdrop[eng.level.long()] if eng.level is not None
                else eng.backdrop.expand(B, H, pitch)).contiguous()
    z = torch.tensor([ord(c) for c in eng.game.z_order], dtype=torch.uint8, device=dev)
    z = z[None].repeat(B, 1).contiguous()
    out = torch.zeros((B, H, pitch), dtype=torch.uint8, device=dev)
    sets.append((eng, backdrop, curtains, z, out))
  cur_stream = lambda: C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
  stream = cur_stream()

  def launch(i):
    eng, backdrop, curtains, z, out = sets[i % len(sets)]
    _lib.check(lib.pcl_render(eng._h, backdrop.data_ptr(), eng.rows * eng.pitch,
                              curtains.data_ptr(), eng.sprites.data_ptr(), z.data_ptr(),
                              out.data_ptr(), cur_stream()), 'pcl_render')   # the capture stream
  for i in range(2 * len(sets)):
    launch(i)
  torch.cuda.synchronize(dev)
  # n launches as one CUDA graph (like the step kernel's timed region): the host
  # cannot feed 15 us kernels one ctypes call at a time without gaps.
  timed = Timed(torch, dev, launch, 0, n)
  timed.run()
  ms = timed.time_ms(lambda: torch.cuda.synchronize(dev)) / n
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  for eng, _, _, _, out in sets:
    assert bool((out[:, :, :eng.cols] == eng.board).all()), 'pcl_render != step kernel board'
  # What a plain elementwise library kernel reaches at THIS launch size with the SAME
  # traffic mix: torch.addcmul(a, b, c, out=o) on u8 planes reads 3 planes and writes 1
  # per env, like the renderer (backdrop + 2 curtains -> board); rotating buffers, same
  # graph timing.  MEASURED_PEAKS' figure is a 4 GB copy; a 67 MB launch whose reads
  # cannot hide behind L2-absorbed writes does not get there.
  copy_ms = None
  try:
    planes = [(s_[1].view(-1), s_[2].view(-1)) for s_ in sets]   # backdrop, 2 curtains
    outs = [torch.empty_like(x[0]) for x in planes]
    half = planes[0][0].numel()
    def ref3to1(i):
      k = i % len(sets)
      bd, cu = planes[k]
      torch.addcmul(bd, cu[:half], cu[half:], out=outs[k])
    tc = Timed(torch, dev, ref3to1, 0, n)
    tc.run()
    copy_ms = tc.time_ms(lambda: torch.cuda.synchronize(dev)) / n
    del outs
  except Exception:                 # noqa: BLE001 - a reference figure only
    copy_ms = None

  # The same kernel over all R batches in ONE launch (R x 4096 envs): how much of
  # the 4096-env figure is launch ramp/tail rather than bandwidth.
  big = None
  try:
    eng0 = sets[0][0]
    BB = sum(s[0].batch for s in sets)
    spec = _lib.Spec()
    spec.abi_version, spec.program = _lib.ABI_VERSION, _lib.PROG_NONE
    spec.rows, spec.cols, spec.pitch = eng0.rows, eng0.cols, eng0.pitch
    spec.n_sprites, spec.n_drapes = len(eng0.sprite_chars), len(eng0.drape_chars)
    for i, ch in enumerate(eng0.sprite_chars):
      spec.sprite_char[i] = ord(ch)
    for i, ch in enumerate(eng0.drape_chars):
      spec.drape_char[i] = ord(ch)
    handle = C.c_void_p()
    _lib.check(lib.pcl_create(C.byref(spec), BB, dev.index, C.byref(handle)), 'pcl_create')
    cat = lambda k: torch.cat([s[k] for s in sets]).contiguous()
    backdrop, curtains, z = cat(1), cat(2), cat(3)
    sprites = torch.cat([s[0].sprites for s in sets]).contiguous()
    out = torch.zeros((BB, eng0.rows, eng0.pitch), dtype=torch.uint8, device=dev)
    def launch_big():
      _lib.check(lib.pcl_render(handle, backdrop.data_ptr(), eng0.rows * eng0.pitch,
                                curtains.data_ptr(), sprites.data_ptr(), z.data_ptr(),
                                out.data_ptr(), stream), 'pcl_render')
    for _ in range(3):
      launch_big()
    torch.cuda.synchronize(dev)
    a.record()
    for _ in range(10):
      launch_big()
    b.record()
    torch.cuda.synchronize(dev)
    big = {'batch': BB, 'kernel_ms_mean': float(a.elapsed_time(b)) / 10}
    lib.pcl_destroy(handle)
  except Exception as e:            # the headline numbers do not depend on this
    big = {'error': str(e)}
  if big is not None:
    big['torch_addcmul_3_planes_in_1_out_ms_4096'] = copy_ms
  return ms, big


def render_roofline(ms, B, eng, peak):
  # A_render = H*W*(2 + D) + 12*S  (SURVEY.md §8d): 16 432 B per env at 64x64, D=2, S=4.
  a_render = eng.rows * eng.cols * 4 + 12 * 4
  achieved = B * a_render / (ms / 1000.0) / 1e9
  return {'kernel': 'render_kernel', 'bound': 'hbm', 'achieved': achieved, 'peak': peak,
          'unit': 'GB/s', 'frac': achieved / peak, 'kernel_ms_mean': ms,
          'algorithmic_bytes_per_launch': B * a_render, 'traffic': None,
          'checked': 'output equals the fused step kernel\'s board'}


def render_big_roofline(big, eng, peak):
  if not big or 'kernel_ms_mean' not in big:
    return big
  a_render = eng.rows * eng.cols * 4 + 12 * 4
  achieved = big['batch'] * a_render / (big['kernel_ms_mean'] / 1000.0) / 1e9
  return dict(big, achieved=achieved, frac=achieved / peak)


def workload_config(n_gpus):
  return {'workload': 'scrolly_maze 64x64 board / 129x129 world, generated levels '
                      '(BASELINE.json configs[1]), random actions 0-4, auto-reset',
          'batch_per_gpu': BATCH_PER_GPU, 'global_batch': BATCH_PER_GPU * n_gpus,
          'levels': N_LEVELS, 'parallelism': 'env-sharded x%d, no collective' % n_gpus,
          'l2': '%d independent %d-env batches stepped round-robin; working set '
                '(~%d MB) exceeds the 126 MB L2, so no flush is needed' % (
                    ROTATION, BATCH_PER_GPU, ROTATION * 60)}


# ------------------------------------------------- the other BASELINE configs

def other_config(name, torch, dist, dev, rank, world, barrier, peak, K):
  """One of BASELINE.json configs[2..4] at this rank's share, timed like the
  headline: graph of K steps over R rotating batches, e2e through the pipelined
  host entry point, roofline of its step kernel, a sampled oracle check."""
  from pycolab_b200 import batched, levels, lowering
  from oracle import engine_model as em
  from oracle import games as ogames
  from oracle import sampled_check
  local = dev.index
  crop_spec = None
  if name == 'C3_warehouse80':
    from pycolab_b200.games import warehouse_manager as g
    arts = [levels.warehouse_level(100 + i) for i in range(16)]
    games = [lowering.lower(g.make_game(a)) for a in arts]
    B, R, n_act = 8192, 3, 4
    a_step, kernel = 80 * 80 * 3 + 64 * 11 + 64, 'warehouse_step'
    what = 'warehouse_manager 80x80, 10 boxes, 16 generated levels, 8192 envs per GPU (configs[2])'
    make = lambda e: ogames.make_warehouse(arts[e % 16])
    sprite_chars = None
  elif name == 'C4_marauders':
    from pycolab_b200.games import extraterrestrial_marauders as g
    art = levels.marauders_level()
    games = [lowering.lower(g.make_game(art))]
    B, R, n_act = 4096, 2, 4
    a_step, kernel = 16 * 39 * 6 + 64 * 7 + 64, 'marauders_step'
    what = ('extraterrestrial_marauders stock 16x39, per-env MT19937, 4096 envs per GPU '
            '(configs[3] = 16384 over 4 GPUs)')
    rngs = {}
    def make(e):                  # one MT19937 stream per env, surviving auto-resets
      if e not in rngs:
        rngs[e] = np.random.RandomState(7 + e)
      return ogames.make_marauders(art, rngs[e])
    sprite_chars = 'Pabcdyz'
  else:
    from pycolab_b200.games import scrolly_maze as g
    arts = [levels.scrolly_maze_level(1000 + i) for i in range(N_LEVELS)]
    games = [lowering.lower(g.make_game(*a)) for a in arts]
    B, R, n_act = 8192, 3, 5
    a_step, kernel = A_STEP_BYTES + 81, 'scrolly_maze_step with the cropper as its epilogue'
    what = ('scrolly_maze 64x64 + ScrollingCropper 9x9 egocentric, 8192 envs per GPU '
            '(configs[4] = 65536 over 8 GPUs)')
    crop_spec = batched.scrolling_crop_spec(9, 9, 0, pad_char=' ', scroll_margins=(None, None))
    make = lambda e: ogames.make_scrolly_maze(arts[e % N_LEVELS][0], arts[e % N_LEVELS][1], '+',
                                              arts[e % N_LEVELS][2])
    sprite_chars = 'Pabc'
  W = 3 * R
  base = rank * R * B
  engines = [batched.BatchedEngine(games, batch=B, device=local, env_offset=base + r * B,
                                   rng_seed=7) for r in range(R)]
  rng0 = [None if e.rng is None else e.rng.clone() for e in engines]   # before any draw
  for e in engines:
    e.its_showtime()
  rs = np.random.RandomState(4321 + rank)
  acts_np = rs.randint(0, n_act, size=(W + K, B)).astype(np.int32)
  acts = torch.from_numpy(acts_np).to(dev)
  states = [e.new_crop_state() for e in engines] if crop_spec is not None else None
  crops = [torch.empty((B, 9, 9), dtype=torch.uint8, device=dev) for _ in engines] \
      if crop_spec is not None else None

  fused_crop = False
  if crop_spec is not None and os.environ.get('PCL_BENCH_SEPARATE_CROP') != '1':
    for r, e in enumerate(engines):            # the cropper as the step kernel's epilogue
      e.attach_cropper(crop_spec, state=states[r], out=crops[r])
    fused_crop = all(e._attached[3] for e in engines)

  def step(t):
    e = engines[t % R]
    e.play(acts[t])
    if crop_spec is not None and e._attached is None:
      e.crop(crop_spec, state=states[t % R], out=crops[t % R])

  l0 = sum(e.launch_count() for e in engines)
  timed = Timed(torch, dev, step, W, K)
  per_step_launches = (sum(e.launch_count() for e in engines) - l0) / float(W + K) \
      if timed.graphs else (2 if crop_spec is not None and not fused_crop else 1)
  ramp_clocks(torch, dev, timed, 0.15)
  for e, r0 in zip(engines, rng0):
    if r0 is not None:
      e.rng.copy_(r0)             # the ramp consumed random draws: rewind the streams
    e.reset()
  if states is not None:
    for s in states:
      s.zero_()
  timed.warm()
  ms_local = timed.time_ms(barrier) / K
  ms, per_rank = max_over_ranks(torch, dist, dev, world, ms_local)
  # oracle replay of a few benchmarked envs (their own level + action stream)
  parity = None
  if make is not None:
    ids = sorted(set(int(i) for i in np.random.RandomState(9).choice(B, 6, replace=False)))
    n = 0
    for r, eng in enumerate(engines[:2]):
      streams = {e: [int(acts_np[t, e]) for t in range(W + K) if t % R == r] for e in ids}
      n += sampled_check.final_state_check(eng, lambda e: make(base + r * B + e), ids, streams,
                                           sprite_chars or '')
    parity = {'envs': 2 * len(ids), 'env_steps': n, 'vs': 'oracle replay, final state identical'}
  crop_checked = None
  if crop_spec is not None and fused_crop:
    # the epilogue's views against the stand-alone crop kernel on the same boards (a
    # perfectly egocentric window depends on the current position only: fresh state)
    crop_checked = all(bool((crops[r] == e.crop(crop_spec, state=e.new_crop_state())).all())
                       for r, e in enumerate(engines))
    assert crop_checked, 'attached cropper != crop_kernel'
  # end to end
  n_e2e = max(2 * R, min(K, 60))
  secs, _ = e2e_pipelined(torch, dev, engines, acts_np, n_e2e, barrier, crop_spec, states)
  secs, _ = max_over_ranks(torch, dist, dev, world, secs)
  eng = engines[0]
  d2h = B * ((81 if crop_spec is not None else eng.rows * eng.pitch) + 10)
  achieved = B * a_step / (ms / 1000.0) / 1e9
  errors = max(int(e.error_codes().abs().max()) for e in engines)
  out = {'workload': what, 'batch_per_gpu': B, 'global_batch': B * world, 'rotation': R,
         'value': world * B / (ms / 1000.0), 'unit': 'env-steps/s', 'ms_per_step': ms,
         'steps': K, 'launches_per_step': per_step_launches, 'launch_path': timed.path,
         'e2e': {'value': world * B * n_e2e / secs, 'unit': 'env-steps/s', 'steps': n_e2e,
                 'h2d_bytes_per_step': B * 4, 'd2h_bytes_per_step': d2h},
         'roofline': {'kernel': kernel, 'bound': 'hbm' if name != 'C4_marauders' else 'latency',
                      'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                      'algorithmic_bytes_per_launch': B * a_step,
                      'note': 'SURVEY 8d reference-layout bytes; static level data is shared '
                              'per level here, so frac may exceed what DRAM actually moves'},
         'parity_checked': parity, 'env_errors': errors}
  if crop_spec is not None:
    out['cropper'] = ('epilogue of the step kernel (pcl_attach_cropper)' if fused_crop
                      else 'separate crop_kernel launch')
    out['crop_checked'] = crop_checked
  for e in engines:
    e.close()
  del engines
  torch.cuda.empty_cache()
  return out


# --------------------------------------------------------------------- main

def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=1000)
  ap.add_argument('--warmup', type=int, default=50)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--cpu-seconds', type=float, default=12.0)
  ap.add_argument('--no-rotate', action='store_true')
  ap.add_argument('--no-configs', action='store_true',
                  help='skip the C3/C4/C5 block (headline only)')
  ap.add_argument('--levels', default='shared', choices=['shared', 'per-env'],
                  help='static level data: one copy per level (default) or one per env')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write what the last timed step returned (rank 0) as DIR/<name>.npy')
  args = ap.parse_args()
  if args.dump_outputs and args.impl == 'reference':
    ap.error('--dump-outputs writes what the device step returned; --impl reference has none')

  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))

  if args.impl == 'reference':
    run_reference_arm(args, rank, world)
    return
  # stdout carries exactly one JSON line: route everything else written to fd 1
  # (e.g. NCCL's version banner, printed from C) to stderr and keep the real
  # stdout for the final line.
  sys.stdout.flush()
  real_stdout = os.fdopen(os.dup(1), 'w')
  os.dup2(2, 1)

  import torch
  import torch.distributed as dist
  from pycolab_b200 import batched
  from pycolab_b200.games import scrolly_maze
  from oracle import games as ogames          # checker for `parity_checked` only
  from oracle import sampled_check

  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  numa = 'off (PCL_BENCH_NUMA_PIN=0)'
  if os.environ.get('PCL_BENCH_NUMA_PIN', '1') != '0':
    numa = pin_to_gpu_numa_node(torch, local_rank, world)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)

  # One poller for the whole job (rank 0 watches every GPU of the box).
  sampler = ClockSampler(','.join(str(i) for i in range(world)) if world > 1 else local_rank)
  if rank == 0:
    sampler.start()
  B, K, W = BATCH_PER_GPU, args.steps, max(3, args.warmup)
  R = 1 if args.no_rotate else ROTATION
  arts = make_levels(N_LEVELS)
  games = [scrolly_maze.make_game(*a) for a in arts]
  from pycolab_b200 import lowering
  lowered = [lowering.lower(g) for g in games]
  # R independent batches of B envs, stepped round-robin: the combined working
  # set (R x ~60 MB) exceeds the 126 MB L2, so every step streams from HBM.
  base = rank * R * B
  engines = [batched.BatchedEngine(lowered, batch=B, device=local_rank,
                                   env_offset=base + r * B) for r in range(R)]
  for e in engines:
    e.its_showtime()
  eng = engines[0]
  rs = np.random.RandomState(1234 + rank)
  actions_np = rs.randint(0, ACTIONS, size=(W + K, B)).astype(np.int32)
  actions = torch.from_numpy(actions_np).to(dev)

  def barrier():
    torch.cuda.synchronize(dev)
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize(dev)

  # ---- device-resident throughput: K steps = one graph replay, one event pair
  timed = Timed(torch, dev, lambda t: engines[t % R].play(actions[t]), W, K)
  ramp_clocks(torch, dev, timed, 0.5)
  for e in engines:                 # clean slate: the oracle replays from its_showtime()
    e.reset()
  sampler.mark_begin()
  timed.warm()
  wall0 = time.perf_counter()
  l_before = sum(e.launch_count() for e in engines)
  dev_ms_local = timed.time_ms(barrier)
  wall = time.perf_counter() - wall0
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, engines[(W + K - 1) % R])
  launches = K if timed.graphs else sum(e.launch_count() for e in engines) - l_before
  dev_ms, per_rank_ms = max_over_ranks(torch, dist, dev, world, dev_ms_local)
  value = world * B * K / (dev_ms / 1000.0)
  kernel_ms = dev_ms / K

  # ---- parity of the BENCHMARKED envs: oracle replay of a sample ------------
  level_of = lambda e: arts[e % N_LEVELS]
  make_world = lambda e: ogames.make_scrolly_maze(level_of(e)[0], level_of(e)[1], '+',
                                                  level_of(e)[2])
  ids = sorted(set(int(i) for i in np.random.RandomState(77 + rank).choice(
      B, max(2, PARITY_ENVS // R), replace=False)))
  parity_steps, t_par = 0, time.perf_counter()
  for r, e_r in enumerate(engines):
    streams = {e: [int(actions_np[t, e]) for t in range(W) if t % R == r] +
                  [int(actions_np[W + t, e]) for t in range(K) if (W + t) % R == r]
               for e in ids}
    parity_steps += sampled_check.final_state_check(
        e_r, lambda e, r=r: make_world(base + r * B + e), ids, streams, 'Pabc')
  parity = {'envs': len(ids) * R, 'steps': (W + K) // R, 'env_steps': parity_steps,
            'vs': 'oracle replay of each sampled env (own level, own action stream, auto-reset): '
                  'final board, reward, discount, done and sprite positions identical',
            'seconds': time.perf_counter() - t_par}
  # ... and in lockstep, every step, on batch 0 (un-timed continuation)
  lock_T = 40
  lock_actions = np.random.RandomState(99 + rank).randint(0, ACTIONS, size=(lock_T, B)).astype(np.int32)
  engines[0].reset()
  parity['lockstep'] = {
      'envs': 16, 'steps': lock_T,
      'compared': sampled_check.lockstep(engines[0], lambda e: make_world(base + e),
                                         ids[:16], lock_actions)}

  # ---- optional hand-off (SURVEY 8e) ---------------------------------------
  handoff = None
  if world > 1:
    handoff = handoff_bench(torch, dist, dev, rank, world, engines, actions, W, K, barrier)

  # Per-launch event timing with an explicit L2 flush before each launch, for
  # comparison (each event pair adds a few microseconds of launch/drain latency).
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
  ev_ms = []
  for t in range(min(K, 50)):
    flush.fill_(t & 0xff)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    eng.play(actions[W + t])
    b.record()
    torch.cuda.synchronize(dev)
    ev_ms.append(a.elapsed_time(b))
  kernel_ms_flushed_events = float(np.median(ev_ms))
  del flush

  # ---- end to end through the host-buffer C-ABI calls ---------------------
  e2e_steps = max(2 * R, min(K, 300))
  e2e_s, _ = e2e_pipelined(torch, dev, engines, actions_np[W:], e2e_steps, barrier)
  e2e_s, e2e_per_rank = max_over_ranks(torch, dist, dev, world, e2e_s)
  e2e_value = world * B * e2e_steps / e2e_s
  # the synchronous single-call form, for comparison
  barrier()
  t0 = time.perf_counter()
  n_sync = max(R, min(K, 40))
  for t in range(n_sync):
    engines[t % R].play_host(actions_np[W + t % K])
  barrier()
  sync_s, _ = max_over_ranks(torch, dist, dev, world, time.perf_counter() - t0)
  pcie, pcie_ranks = None, None
  try:
    g = pcie_probe(torch, dev, barrier)
    if world > 1:
      t = torch.tensor([g], device=dev, dtype=torch.float64)
      every = [torch.zeros_like(t) for _ in range(world)]
      dist.all_gather(every, t)
      pcie_ranks = [round(float(v.item()), 2) for v in every]
    pcie = g
  except Exception:               # noqa: BLE001 - informational
    pass
  render_ms, render_big = render_microbench(engines, n=60) if rank == 0 else (None, None)
  sampler.mark_end()
  clocks = sampler.stop() if rank == 0 else None
  errors = max(int(e.error_codes().abs().max()) for e in engines)

  peaks = {}
  try:
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
  except (OSError, ValueError):
    pass
  peak = float(peaks.get('hbm_gbs', 6650.0))

  # ---- per-env level copies: the second data point (no level sharing) -------
  per_env_levels = None
  if not args.no_configs:
    try:
      per_env_levels = per_env_level_point(torch, dist, dev, world, rank, lowered, actions, W, K,
                                           barrier, peak)
    except Exception as err:      # noqa: BLE001 - informational
      per_env_levels = {'error': str(err)[:200]}

  # ---- the other BASELINE configs -------------------------------------------
  for e in engines[1:]:
    e.close()
  configs = {}
  if not args.no_configs:
    kc = max(6, min(K, 240))
    for name in ('C3_warehouse80', 'C4_marauders', 'C5_scrolly64_crop9'):
      try:
        configs[name] = other_config(name, torch, dist, dev, rank, world, barrier, peak, kc)
      except Exception as err:    # noqa: BLE001 - the headline line must still print
        configs[name] = {'error': '%s: %s' % (type(err).__name__, str(err)[:200])}

  if rank == 0:
    traffic = {}
    try:
      traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
    except (OSError, ValueError):
      pass
    achieved = B * A_STEP_BYTES / (kernel_ms / 1000.0) / 1e9
    layout = B * LAYOUT_STEP_BYTES / (kernel_ms / 1000.0) / 1e9
    dram = B * DRAM_STEP_BYTES / (kernel_ms / 1000.0) / 1e9
    kind = cpu_kind()
    cpu_value, cpu_steps = cpu_baseline(1, args.cpu_seconds, kind)
    real_stdout.write(json.dumps({
        'metric': 'env_steps_per_sec', 'value': value, 'unit': 'env-steps/s',
        'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': dev_ms / K,
        'per_rank_ms_per_step': [m / K for m in per_rank_ms],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'u8', 'data': 'synthetic', 'config': workload_config(world),
        'clocks': clocks, 'gpu_launches': launches, 'launch_path': timed.path,
        'numa': numa, 'parity_checked': parity,
        'e2e': {'value': e2e_value, 'unit': 'env-steps/s', 'steps': e2e_steps,
                'h2d_bytes_per_step': B * 4,
                'd2h_bytes_per_step': B * (BOARD[0] * eng.pitch + 4 + 1 + 4 + 1),
                'path': 'pcl_step_host_async + pcl_host_wait, 2 steps in flight over the '
                        'rotating batches, pinned host buffers',
                'per_rank_seconds': e2e_per_rank,
                'sync_call_value': world * B * n_sync / sync_s,
                'sync_call_path': 'pcl_step_host (one blocking call per step)',
                'pcie_d2h_gbs_this_rank': pcie, 'pcie_d2h_gbs_per_rank': pcie_ranks,
                'pcie_bound_value': None if not pcie else
                    world * (min(pcie_ranks) if pcie_ranks else pcie) * 1e9 /
                    (BOARD[0] * eng.pitch + 14)},
        'roofline': {
            'kernel': 'scrolly_maze_step', 'bound': 'hbm',
            # primary: the bytes THIS layout moves through DRAM per env-step
            'achieved': layout, 'peak': peak, 'unit': 'GB/s', 'frac': layout / peak,
            'bytes_per_launch': B * LAYOUT_STEP_BYTES,
            'peak_source': 'MEASURED_PEAKS.json' if peaks else 'fallback 6650',
            'kernel_ms_mean': kernel_ms,
            'kernel_ms_flushed_event_pairs_median': kernel_ms_flushed_events,
            'traffic': traffic.get('scrolly_maze_step', {}).get('bytes'),
            'traffic_source': traffic.get('scrolly_maze_step', {}).get('source'),
            # secondary: SURVEY 8d's reference-layout count (can exceed 1: static level
            # data is stored once per level and served from L2, curtains are bit-packed)
            'dram_bytes_per_launch': B * DRAM_STEP_BYTES, 'dram_achieved': dram,
            'dram_frac': dram / peak,
            'survey_bytes_per_launch': B * A_STEP_BYTES,
            'survey_achieved': achieved, 'survey_frac': achieved / peak,
            'note': 'frac = the bytes this layout moves per env-step (backdrop tile 4096 + board '
                    '4096 + two bit-packed windows 1024 + records 512 = 9 728) / time / measured '
                    'copy peak; dram_* counts only what must reach DRAM with shared levels (board '
                    '4096 + coin window sectors 2048 + records 512); survey_* uses the '
                    'reference-layout 24 896 B per env-step of SURVEY 8d, which also counts byte '
                    'curtains this engine never materialises',
            'per_env_levels': per_env_levels},
        'cpu_baseline': {'value': cpu_value, 'unit': 'env-steps/s', 'cores': 1,
                         'kind': kind, 'what': cpu_note(kind),
                         'usable_cores_on_this_box': usable_cores(),
                         'sample': '%d env-steps of one env on the same generated '
                                   '64x64 levels' % cpu_steps},
        'render_roofline': dict(render_roofline(render_ms, B, eng, peak),
                                traffic=traffic.get('render_kernel', {}).get('bytes'),
                                one_launch_over_all_batches=render_big_roofline(
                                    render_big, eng, peak)),
        'handoff_allgather': handoff, 'configs': configs,
        'wall_s_timed_region': wall, 'env_errors': errors}) + "\n")
    real_stdout.flush()
  if world > 1:
    dist.destroy_process_group()


DUMP_BOARDS = 1024                # envs whose boards --dump-outputs writes (16 MB as f32)


def dump_outputs(path, eng):
  """The StepResult of `eng`'s last step as float32 .npy files: reward, has_reward,
  discount and done of every env, and the boards of a fixed, seeded sample of
  DUMP_BOARDS envs (all B boards as float32 would be 64 MB) with their indices."""
  os.makedirs(path, exist_ok=True)
  envs = np.sort(np.random.RandomState(0).choice(eng.batch, min(DUMP_BOARDS, eng.batch),
                                                 replace=False))
  arrays = {'board_sample': eng.board.cpu().numpy()[envs], 'board_sample_env': envs,
            'reward': eng.reward.cpu().numpy(), 'has_reward': eng.has_reward.cpu().numpy(),
            'discount': eng.discount.cpu().numpy(), 'done': eng.done.cpu().numpy()}
  for name, a in arrays.items():
    np.save(os.path.join(path, name + '.npy'), a.astype(np.float32))


def per_env_level_point(torch, dist, dev, world, rank, lowered, actions, W, K, barrier, peak):
  """The headline step with one copy of the static level data PER ENV (no sharing
  through `d_level`): backdrop + wall pattern then stream from HBM too."""
  from pycolab_b200 import batched
  B, R = BATCH_PER_GPU, 3
  engines = [batched.BatchedEngine(lowered, batch=B, device=dev.index, share_levels=False,
                                   env_offset=(rank * R + r) * B) for r in range(R)]
  for e in engines:
    e.its_showtime()
  kk = max(6, min(K, 120))
  timed = Timed(torch, dev, lambda t: engines[t % R].play(actions[t % (W + K)]), 3, kk)
  timed.warm()
  timed.run()
  ms = timed.time_ms(barrier) / kk
  ms, _ = max_over_ranks(torch, dist, dev, world, ms)
  per_env_bytes = DRAM_STEP_BYTES + 4096 + 64 * 32
  out = {'kernel_ms_mean': ms, 'value': world * B / (ms / 1000.0),
         'bytes_per_launch': B * per_env_bytes,
         'achieved': B * per_env_bytes / (ms / 1000.0) / 1e9,
         'frac': B * per_env_bytes / (ms / 1000.0) / 1e9 / peak,
         'note': 'DRAM bytes with one copy of the level data per env: board 4096 + coin window '
                 'sectors 2048 + records 512 + backdrop tile 4096 + wall window sectors 2048'}
  for e in engines:
    e.close()
  return out


def handoff_bench(torch, dist, dev, rank, world, engines, actions, W, K, barrier):
  """Every rank receives every shard's egocentric 9x9 crop + reward / discount /
  done each step.  Times step + hand-off (ONE kernel after the step: cropper, record
  packing, stores into every rank's gather buffer over NVLink, flag barrier) as a
  CUDA graph, and checks the result against a plain NCCL all-gather."""
  from pycolab_b200 import batched
  from pycolab_b200 import dist as pdist
  B, R = engines[0].batch, len(engines)
  spec = batched.scrolling_crop_spec(9, 9, 0, pad_char=' ', scroll_margins=(None, None))
  fused_err = None
  try:
    one_kernel = os.environ.get('PCL_BENCH_HANDOFF_SINGLE_KERNEL') == '1'
    handoffs = [pdist.FusedHandoff(e, spec, world * B, signal_kernel=not one_kernel)
                for e in engines]
    transport = ('crop + pack + %s into symmetric memory in one kernel, %s' % (
        handoffs[0].transport, 'flag barrier in the same kernel' if one_kernel else
        'flags published and awaited by a one-warp kernel behind it'))
    kind = 'fused'
  except Exception as err:      # noqa: BLE001 - any failure to set peer mapping up
    fused_err = str(err).splitlines()[0][:120] if str(err) else type(err).__name__
    kind = 'nccl'
  agree = torch.tensor([0 if kind == 'fused' else 1], device=dev)
  dist.all_reduce(agree, op=dist.ReduceOp.MAX)
  if int(agree.item()):         # some rank cannot map peer memory: all use NCCL
    kind = 'nccl'
    handoffs = [pdist.Handoff(e, (9, 9), world * B) for e in engines]
    transport = 'crop kernel + pack kernel + 1 NCCL all-gather (symmetric memory unavailable: %s)' % (
        fused_err or 'on a peer')
  states = [e.new_crop_state() for e in engines]
  crops = [torch.empty((B, 9, 9), dtype=torch.uint8, device=dev) for _ in engines]

  def step_and_gather(t):
    e = engines[t % R]
    e.play(actions[W + (t % K)])
    if kind == 'fused':
      return handoffs[t % R].gather()
    return handoffs[t % R].gather(e.crop(spec, state=states[t % R], out=crops[t % R]))

  n_h = max(2 * R, (min(K, 120) // (2 * R)) * 2 * R)     # even number of calls per batch
  for t in range(2 * R):
    step_and_gather(t)
  barrier()
  timed = Timed(torch, dev, step_and_gather, 0, n_h) if kind == 'fused' else None
  if timed is not None and timed.graphs:
    timed.run()                                           # upload + first replay, untimed
    ms_local = timed.time_ms(barrier) / n_h
    path = timed.path
  else:
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    h0.record()
    for t in range(n_h):
      step_and_gather(t)
    h1.record()
    barrier()
    ms_local = float(h0.elapsed_time(h1)) / n_h
    path = 'host loop'
  ms, per_rank = max_over_ranks(torch, dist, dev, world, ms_local)
  # correctness of the timed transport: one more step through it, and the same
  # step's tensors through the stand-alone cropper + plain NCCL all-gathers
  barrier()
  gathered = step_and_gather(0)
  e = engines[0]
  mine = e.crop(spec, state=states[0], out=crops[0])
  want = pdist.allgather_outputs([mine, e.reward, e.discount, e.done, e.has_reward], world * B)
  ok = all(bool((g == w).all()) for g, w in zip(gathered, want))
  if kind == 'fused':           # keep every batch at an even number of fused calls
    step_and_gather(0)
  flag = torch.tensor([1 if ok else 0], device=dev)
  dist.all_reduce(flag, op=dist.ReduceOp.MIN)
  rec = handoffs[0].rec if kind == 'fused' else pdist.handoff_record_bytes(81)
  # ---- split phase (lag 1): signal this step, wait only for the previous one ----------
  split = None
  if kind == 'fused':
    try:
      lagged = [pdist.FusedHandoff(e, spec, world * B, lag=1, signal_kernel=not one_kernel)
                for e in engines]

      def step_and_send(t):
        engines[t % R].play(actions[W + (t % K)])
        return lagged[t % R].gather()
      for t in range(2 * R):
        step_and_send(t)
      barrier()
      timed2 = Timed(torch, dev, step_and_send, 0, n_h)
      if timed2.graphs:
        timed2.run()
        ms2_local = timed2.time_ms(barrier) / n_h
        ms2, per_rank2 = max_over_ranks(torch, dist, dev, world, ms2_local)
        # correctness: one more step outside the graph; after flush() the records of that
        # step equal the stand-alone cropper + NCCL all-gather, on every rank
        barrier()
        step_and_send(0)
        got = lagged[0].flush()
        e0 = engines[0]
        mine2 = e0.crop(spec, state=e0.new_crop_state())        # egocentric: position only
        want2 = pdist.allgather_outputs([mine2, e0.reward, e0.discount, e0.done, e0.has_reward],
                                        world * B)
        ok2 = all(bool((g == w).all()) for g, w in zip(got, want2))
        flag2 = torch.tensor([1 if ok2 else 0], device=dev)
        dist.all_reduce(flag2, op=dist.ReduceOp.MIN)
        split = {'what': 'the same hand-off, split phase: the kernel of step t signals t and waits '
                         'only for step t - 1 of the peers (three buffer parts), consumers read one '
                         'step behind, a host barrier completes the last step',
                 'ms_per_step': ms2, 'per_rank_ms_per_step': per_rank2, 'steps': n_h,
                 'value': world * B / (ms2 / 1000.0), 'unit': 'env-steps/s',
                 'handoff_checked': bool(int(flag2.item()))}
    except Exception as err:        # noqa: BLE001 - the strict figure above stands on its own
      split = {'error': str(err).splitlines()[0][:160] if str(err) else type(err).__name__}
  return {'split_phase': split,
          'what': 'step + 9x9 crop + hand-off of the packed (crop, reward, discount, done) '
                  'records to every rank', 'transport': transport, 'launch_path': path,
          'ms_per_step': ms, 'per_rank_ms_per_step': per_rank, 'steps': n_h,
          'value': world * B / (ms / 1000.0), 'unit': 'env-steps/s',
          'handoff_checked': bool(int(flag.item())),
          'checked_against': 'stand-alone crop kernel + dist.all_gather_into_tensor of '
                             'crop/reward/discount/done/has_reward of the same step, every rank',
          'record_bytes': rec,
          'nvlink_bytes_in_per_rank_per_step': (world - 1) * B * rec}


if __name__ == '__main__':
  main()
