"""Benchmark of the hot path: env-steps/s (= rendered frames/s) of step+render.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4|c5]
    python bench.py --impl reference ...      # the CPU path (oracle port) on the host cores

One "step" = one Environment.step (action -> pose/velocity update -> reward ->
termination/auto-reset -> PILRenderer frame) for every env of the batch.  Prints ONE JSON
line (rank 0).  See DESIGN.md "Measurement" for what each key means.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'env_steps_per_sec'
UNIT = 'env-steps/s'


def _peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      return float(json.load(f)['hbm_gbs']), 'measured'
  return 6650.0, 'fallback'


class ClockSampler(threading.Thread):
  """nvidia-smi SM clock / throttle-reason samples during the timed region."""
  Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index, self.rows, self.proc = index, [], None

  def run(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
           '--format=csv,noheader,nounits', '-lms', '100'],
          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      for line in self.proc.stdout:
        self.rows.append([c.strip() for c in line.split(',')])
    except Exception:
      pass

  def stop(self):
    if self.proc is not None:
      self.proc.terminate()
    self.join(timeout=2)
    sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
    mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
    reasons = set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for r in self.rows:
      for n, v in zip(names, r[3:7]):
        if v == 'Active':
          reasons.add(n)
    return dict(sm_mhz=float(np.median(sm)) if sm else None,
                sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons),
                samples=len(sm))


def usable_cores():
  """Host CPUs this process may actually use: the affinity mask capped by the cgroup CPU
  quota (cpu.max).  On the GPU boxes 128 logical CPUs are visible but the container's quota
  is 16; more threads than that only add throttling."""
  try:
    n = len(os.sched_getaffinity(0))
  except AttributeError:
    n = os.cpu_count() or 1
  quota = None
  try:   # cgroup v2
    with open('/sys/fs/cgroup/cpu.max') as f:
      q, period = f.read().split()[:2]
    if q != 'max':
      quota = int(q) / float(period)
  except (OSError, ValueError):
    try:   # cgroup v1
      with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
        q = int(f.read())
      with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
        period = int(f.read())
      if q > 0 and period > 0:
        quota = q / float(period)
    except (OSError, ValueError):
      pass
  if quota:
    n = max(1, min(n, int(round(quota))))
  return n


def cpu_reference(wl, n_sample_envs, steps, warmup, seed=1000, cores=None):
  """The reference's algorithm on the host cores: oracle port (C restatement of the
  reference path incl. Pillow's polygon fill and LANCZOS), one thread per core, each
  stepping its own slice of a bounded env sample.  Returns (env-steps/s, cores, seconds)."""
  from concurrent.futures import ThreadPoolExecutor
  from oracle import oracle
  from spriteworld_b200 import constants
  from tests import fixtures
  cores = cores or usable_cores()
  n = max(cores, (n_sample_envs // cores) * cores)
  K = max(2, (steps + warmup) // wl.max_episode_length + 2)
  rng = np.random.RandomState(seed)
  scenes = wl.sample_scenes(rng, n * K)
  rec = np.zeros((n * K, wl.n_slots), oracle.SPRITE_DTYPE)
  for f in ('x', 'y', 'm00', 'm01', 'm10', 'm11', 'vx', 'vy', 'member', 'shape', 'pos_f32', 'rgb'):
    rec[f] = scenes[f]
  pool = rec.reshape(n, K, wl.n_slots)
  cfg = fixtures.env_cfg_from_meta(dict(
      action=wl.action, keep_in_frame=True, max_episode_length=wl.max_episode_length,
      nodes=[dict(n, goal=list(n.get('goal', (0, 0))), weights=list(n.get('weights', (1, 1))))
             if n['kind'] == 'find_goal' else n for n in wl.nodes]))
  tab = oracle.shape_table(constants.SHAPES)
  rc = oracle.raster_cfg(wl.image_size[0], wl.image_size[1], wl.anti_aliasing)
  bo = oracle.BatchOracle(cfg, tab, rc, pool)
  actions = wl.sample_actions(np.random.RandomState(7), steps + warmup, n)
  chunk = n // cores
  with ThreadPoolExecutor(cores) as ex:
    def one_step(t):
      list(ex.map(lambda c: bo.step(actions[t], c * chunk, (c + 1) * chunk), range(cores)))
    for t in range(warmup):
      one_step(t)
    t0 = time.perf_counter()
    for t in range(warmup, warmup + steps):
      one_step(t)
    dt = time.perf_counter() - t0
  return n * steps / dt, cores, dt, n


def workload_config(wl, envs_per_gpu=None):
  """The keys both arms put into `config` (the driver compares them)."""
  w, h = wl.image_size
  return dict(workload=wl.name, envs_per_gpu=int(envs_per_gpu or wl.n_envs), n_sprites=wl.n_slots,
              image=[h, w, 3], anti_aliasing=wl.anti_aliasing,
              max_episode_length=wl.max_episode_length)


def run_reference_arm(args, wl):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  # each step = a bounded sample of the workload sized to finish within minutes
  n_sample = 128 * usable_cores()
  value, cores, dt, n = cpu_reference(wl, n_sample, args.steps, args.warmup)
  sample = ('%d envs x %d steps of %s on %d host threads = usable cores (cgroup quota; %d logical '
            'CPUs visible), oracle C port of the reference path' % (
                n, args.steps, wl.name, cores, os.cpu_count() or 1))
  cfg = workload_config(wl, args.envs)
  cfg['sample_envs'] = n
  line = dict(
      impl='reference', metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus,
      steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
      higher_is_better=True, scaling='weak', vs_baseline=None, dtype='u8', data='synthetic',
      config=cfg,
      cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind='port', sample=sample),
      e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
  print(json.dumps(line))


def bind_to_gpu_numa_node(local_rank):
  """Pins this process to the CPUs of the NUMA node the GPU hangs off, so that the pinned
  host buffers of the e2e path (first touch) and the copy threads are local to the GPU's
  PCIe root.  Returns the node id or None."""
  try:
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
    bus = pynvml.nvmlDeviceGetPciInfo(h).busId
    bus = bus.decode() if isinstance(bus, bytes) else bus
    bus = bus.lower()
    if len(bus.split(':')[0]) == 8:   # nvml prints an 8-digit domain, sysfs has 4
      bus = bus[4:]
    with open('/sys/bus/pci/devices/%s/numa_node' % bus) as f:
      node = int(f.read())
    if node < 0:
      return None
    with open('/sys/devices/system/node/node%d/cpulist' % node) as f:
      cpus = set()
      for part in f.read().strip().split(','):
        lo, _, hi = part.partition('-')
        cpus.update(range(int(lo), int(hi or lo) + 1))
    cpus &= os.sched_getaffinity(0)
    if cpus:
      os.sched_setaffinity(0, cpus)
      return node
  except Exception:
    pass
  return None


DUMP_BUDGET_BYTES = 60 * 10 ** 6   # the arrays of --dump-outputs; with the .npy headers < 64 MB
DUMP_SEED = 0


def dump_outputs(res, out_dir):
  """Writes the per-env outputs of one step (an engine.StepResult) as DIR/<name>.npy, so that two
  builds can be compared output for output: reward (float64), step_type, success, status and
  frames (float32, exact for their integer values), and env_index (float64), the envs they belong
  to.  When all envs would exceed DUMP_BUDGET_BYTES, the envs are a fixed sample drawn with
  DUMP_SEED, in ascending order."""
  import torch
  os.makedirs(out_dir, exist_ok=True)
  E = int(res.reward.shape[0])
  per_env = 8 * 2 + 4 * (3 + res.frames[0].numel())   # reward, env_index; the float32 arrays
  n = min(E, DUMP_BUDGET_BYTES // per_env)
  idx = np.arange(E) if n == E else np.sort(np.random.RandomState(DUMP_SEED).choice(E, n, replace=False))
  rows = torch.as_tensor(idx, device=res.reward.device)
  arrays = dict(env_index=idx.astype(np.float64))
  for name in ('reward', 'step_type', 'success', 'status', 'frames'):
    a = getattr(res, name).index_select(0, rows).cpu().numpy()
    arrays[name] = a.astype(np.float64 if name == 'reward' else np.float32)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), a)


class Bench(object):
  """One workload on this rank's GPU: engine, frame ring, gather plumbing, timed loops."""

  def __init__(self, wl, args, world, rank, local_rank, steps, warmup, E=None,
               max_episode_length=None):
    import torch
    from spriteworld_b200 import workloads
    self.torch, self.wl, self.args = torch, wl, args
    self.world, self.rank = world, rank
    self.dev = torch.device('cuda', local_rank)
    self.steps, self.warmup = steps, warmup
    self.E = E = E or wl.n_envs          # per GPU: weak scaling by env index
    self.T = T = warmup + steps
    mel = max_episode_length or wl.max_episode_length
    # the action/scene tables cover one block of T steps; longer runs wrap around, and the
    # ring of pooled scenes per env is as deep as the resets of one block need
    self.K = K = min(T // mel + 3, 64)
    self.eng, self.raster, _ = workloads.build_engine(wl, E, K, device=local_rank,
                                                      seed=1000 + rank, max_episode_length=mel)
    self.actions = torch.from_numpy(wl.sample_actions(np.random.RandomState(7 + rank), T, E)).to(self.dev)
    self.H, self.W = wl.image_size[1], wl.image_size[0]
    self.frame_bytes = E * self.H * self.W * 3
    # frame ring larger than L2 (126 MB) so that every step's frame writes reach HBM
    self.n_ring = max(2, int(np.ceil(160e6 / self.frame_bytes)) + 1)
    self.ring = [self.raster.new_frames() for _ in range(self.n_ring)]
    self.gathered, self.peer, self.inflight, self.n_gslots = None, None, [], 2
    self.last = None   # StepResult of the latest step
    self.gather = args.gather
    if world > 1 and self.gather == 'nccl':
      self._nccl_buffers()
    elif world > 1:
      from spriteworld_b200 import _native, distributed
      # as many gathered buffers as make one pass over them larger than L2
      self.n_gslots = max(2, int(np.ceil(160e6 / (world * self.frame_bytes))) + 1)
      try:
        self.peer = distributed.PeerFrames(E, (self.H, self.W, 3), self.dev, n_slots=self.n_gslots)
        # reward / step type / success / status of every rank (11 bytes per env), per gathered slot
        self.out_all = [torch.empty(world * E * 11, dtype=torch.uint8, device=self.dev)
                        for _ in range(self.n_gslots)]
      except _native.NativeError as ex:   # raised on every rank or on none
        if rank == 0:
          sys.stderr.write('peer-memory gather unavailable (%s); using the NCCL all-gather\n' % ex)
        self.gather = 'nccl'
        self._nccl_buffers()

  def _nccl_buffers(self):
    torch = self.torch
    self.gathered = [torch.empty((self.world * self.E, self.H, self.W, 3), dtype=torch.uint8,
                                 device=self.dev) for _ in range(2)]

  def close(self):
    self.drain()
    if self.peer is not None:
      self.peer.close()
    self.raster.close()
    self.eng.close()
    self.ring = self.gathered = None
    self.torch.cuda.empty_cache()

  def wait_for(self, pred):
    for item in list(self.inflight):
      if pred(item):
        item[0].wait()
        self.inflight.remove(item)

  def one_step(self, t, gather=True):
    import torch.distributed as dist
    eng, raster, peer, T = self.eng, self.raster, self.peer, self.T
    slot, dst = t % self.n_ring, t % (self.n_gslots if peer is not None else 2)
    if self.world > 1 and gather and peer is not None:
      # the single collective of the path, fused: the render kernel stores each frame into
      # every rank's gathered buffer over NVLink; a one-element all-reduce on NCCL's stream
      # is the completion barrier and overlaps the next step
      self.wait_for(lambda it: it[2] == dst)   # everyone is done with the step that last used dst
      if self.gather == 'ce':
        # variant: render into this rank's block, then copy-engine pushes to the peers
        self.last = eng.step(self.actions[t % T], raster, peer.own_slab(dst))
        self.inflight.append((peer.push(dst), -1, dst))
      else:
        # the per-env records ride along as ONE all-gather behind the kernel (SURVEY 8e); it is also
        # the completion barrier of the frame stores: it cannot finish before every rank's kernel has
        self.last = eng.step_gather(self.actions[t % T], raster, peer.slot(dst))
        self.inflight.append((dist.all_gather_into_tensor(self.out_all[dst], eng.out_bytes, async_op=True),
                              -1, dst))
      return
    self.wait_for(lambda it: it[1] == slot)    # the gather that last read this ring buffer
    fr = self.ring[slot]
    self.last = eng.step(self.actions[t % T], raster, fr)
    if self.world > 1 and gather:
      # the single collective of the path as a separate NCCL all-gather.  It runs on NCCL's
      # stream and overlaps the next step's compute.
      self.wait_for(lambda it: it[2] == dst)
      self.inflight.append((dist.all_gather_into_tensor(self.gathered[dst], fr, async_op=True), slot, dst))

  def drain(self):
    self.wait_for(lambda it: True)

  def barrier(self):
    self.drain()
    if self.world > 1:
      import torch.distributed as dist
      dist.barrier()
    self.torch.cuda.synchronize()

  def _max_over_ranks(self, ms):
    if self.world > 1:
      import torch.distributed as dist
      t = self.torch.tensor([ms], device=self.dev, dtype=self.torch.float64)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t.item())
    return ms

  def timed_steps(self, gather=True, t_base=0):
    """Exactly `steps` steps, bracketed by barrier + synchronize and timed with CUDA events (max
    over ranks); returns the milliseconds."""
    torch = self.torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    self.barrier()
    ev0.record()
    for t in range(t_base, t_base + self.steps):
      self.one_step(t, gather)
    self.drain()
    ev1.record()
    self.barrier()
    return self._max_over_ranks(ev0.elapsed_time(ev1))

  def run(self, sampler=None, dump_dir=None):
    """Warm-up, the timed steps, the sharded variant at N > 1 and the render kernel alone.
    With `dump_dir`, the outputs of the last timed step are written there (dump_outputs)."""
    torch = self.torch
    if sampler:   # before the warm-up, so that the GPU does not idle right before the timed steps
      sampler.start()
      time.sleep(0.3)
    for t in range(self.warmup):
      self.one_step(t)
    self.barrier()
    launches0 = self.eng.launch_count()
    ms = self.timed_steps(True, self.warmup)
    launches = self.eng.launch_count() - launches0
    res = dict(value=self.world * self.E * self.steps / (ms * 1e-3), ms_per_step=ms / self.steps,
               launches=int(launches), timed=dict(steps=self.steps, seconds=ms * 1e-3))
    if dump_dir:
      # before anything else runs: the render loop below reuses the frame buffers
      dump_outputs(self.last, dump_dir)
    if self.world > 1:
      # SURVEY 8(e) asks for both numbers: the same steps with the frames left sharded
      sms = self.timed_steps(False, self.T)
      res['frames_sharded'] = dict(value=self.world * self.E * self.steps / (sms * 1e-3), unit=UNIT,
                                   ms_per_step=sms / self.steps)
      # the gather's NVLink load: every rank takes in the other ranks' frames each step
      ingest = (self.world - 1) * self.frame_bytes
      res['nvlink'] = dict(ingest_bytes_per_gpu_per_step=int(ingest),
                           achieved_gbs_per_direction_per_gpu=ingest / (ms / self.steps * 1e-3) / 1e9,
                           nominal_gbs_per_direction=900.0)
    # dominant kernel alone: launches of the render kernel, CUDA events on its stream
    evr0, evr1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_r = max(20, min(self.steps, 100))
    for i in range(3):
      self.eng.render(self.raster, self.ring[i % self.n_ring])
    torch.cuda.synchronize()
    evr0.record()
    for i in range(n_r):
      self.eng.render(self.raster, self.ring[i % self.n_ring])
    evr1.record()
    torch.cuda.synchronize()
    res['render_ms'] = evr0.elapsed_time(evr1) / n_r
    return res

  def roofline(self, render_ms, traffic=None):
    peak, peak_kind = _peaks()
    alg_bytes = self.wl.algorithmic_bytes() * self.E
    achieved = alg_bytes / (render_ms * 1e-3) / 1e9
    return dict(bound='hbm', achieved=achieved, peak=peak, unit='GB/s', frac=achieved / peak,
                traffic=traffic, peak_kind=peak_kind, kernel='render_kernel', kernel_ms=render_ms,
                algorithmic_bytes_per_launch=alg_bytes)

  def e2e(self):
    """End to end through the C-ABI with HOST buffers (pinned): H2D actions, D2H frames+outputs."""
    torch, E = self.torch, self.E
    a_host = torch.from_numpy(self.wl.sample_actions(np.random.RandomState(99 + self.rank), 8, E)).pin_memory()
    out = dict(
        frames=torch.empty((E, self.H, self.W, 3), dtype=torch.uint8).pin_memory().numpy(),
        reward=torch.empty(E, dtype=torch.float64).pin_memory().numpy(),
        step_type=torch.empty(E, dtype=torch.int8).pin_memory().numpy(),
        success=torch.empty(E, dtype=torch.uint8).pin_memory().numpy(),
        status=torch.empty(E, dtype=torch.uint8).pin_memory().numpy())
    n_e2e = max(10, min(self.steps, 50))
    a_np = a_host.numpy()
    for i in range(3):
      self.eng.step_host(a_np[i % 8], self.raster, out=out)
    times = []
    for rep in range(20):
      self.barrier()
      t0 = time.perf_counter()
      for i in range(n_e2e):
        self.eng.step_host(a_np[i % 8], self.raster, out=out)
      self.barrier()
      times.append(self._max_over_ranks(1e3 * (time.perf_counter() - t0)) * 1e-3)
      if sum(times) >= 1.0:
        break
    dt = float(np.median(times))
    d2h = int(self.frame_bytes + E * (8 + 1 + 1 + 1))
    return dict(value=self.world * E * n_e2e / dt, unit=UNIT,
                h2d_bytes_per_step=int(a_np[0].nbytes), d2h_bytes_per_step=d2h,
                steps=n_e2e, blocks=len(times), ms_per_step=1e3 * dt / n_e2e,
                d2h_gbs_per_gpu=d2h / (dt / n_e2e) / 1e9,
                path='swb_step_host: pinned host actions -> H2D -> step+render -> D2H frames, '
                     'reward, step_type, success, status -> stream sync')


def _traffic(key):
  """DRAM bytes per render launch from the committed ncu capture (profiles/traffic.json):
  a record, not a live measurement -- ncu cannot run inside the timed process."""
  tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
  if not os.path.exists(tpath):
    return None, None
  with open(tpath) as f:
    d = json.load(f)
  return d.get(key), d.get('source')


def api_rate(wl, E, local_rank, steps):
  """env-steps/s through the Python plugin API: BatchedEnvironment.step with device actions,
  auto-reset from the scene ring and its asynchronous refill (every env resets each
  max_episode_length steps, C2's worst case)."""
  import torch
  from spriteworld_b200 import environment
  env = environment.BatchedEnvironment(n_envs=E, device=local_rank, rng=np.random.RandomState(4242),
                                       pool_depth=32, **wl.plugin_config())
  acts = torch.from_numpy(wl.sample_actions(np.random.RandomState(5), 16, E)).to(env.engine.device)
  for i in range(4 * wl.max_episode_length + 3):
    env.step(acts[i % 16])
  torch.cuda.synchronize()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  n = max(steps, 20 * wl.max_episode_length)
  t0 = time.perf_counter()
  ev0.record()
  for i in range(n):
    env.step(acts[i % 16])
  ev1.record()
  torch.cuda.synchronize()
  wall = time.perf_counter() - t0
  ms = max(ev0.elapsed_time(ev1), 1e3 * wall)
  stats = env.refill_stats()
  env.close()
  return dict(value=E * n / (ms * 1e-3), unit=UNIT, steps=n, ms_per_step=ms / n,
              path='BatchedEnvironment.step (device actions -> BatchedTimeStep on the device); every '
                   'env resets each max_episode_length steps; the scene ring (32 deep) is refilled '
                   'asynchronously: scenes drawn through the plugin API (factor_distributions / '
                   'sprite_generators) by one host thread, uploaded over a side stream',
              host_scenes_per_sec=stats['scenes'] / max(stats['host_seconds'], 1e-9), refill=stats)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=200)
  ap.add_argument('--warmup', type=int, default=20)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--workload', default='c2', choices=['c2', 'c3', 'c4', 'c5'])
  ap.add_argument('--also', default=None,
                  help='comma list of the other BASELINE configs measured in the same run '
                       '(default: c3,c4,c5 at N=1; c4,c5 at N>1; "none" to skip)')
  ap.add_argument('--envs', type=int, default=0, help='override envs per GPU')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write the outputs of the last timed step of the headline workload to '
                       'DIR/<name>.npy (float32 / float64); at N > 1, those of rank 0\'s envs')
  ap.add_argument('--gather', default='peer', choices=['peer', 'ce', 'nccl'],
                  help='N>1 frame gather: stores into peer memory from the render kernel, or a '
                       'separate NCCL all-gather')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-e2e', action='store_true')
  ap.add_argument('--no-api', action='store_true')
  args = ap.parse_args()
  if args.warmup < 3:
    args.warmup = 3
  from spriteworld_b200 import workloads
  wl = workloads.WORKLOADS[args.workload]()
  if args.impl == 'reference':
    return run_reference_arm(args, wl)

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
  import torch
  import torch.distributed as dist
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
  torch.cuda.set_device(local_rank)

  # the plugin-API rate first, in a process that holds nothing else yet: its bound is the host
  # sampler (NumPy), which ran three times slower after the other measurements of this process
  # (pinned buffers, several hundred MB of frame rings) than alone
  api = None
  if world == 1 and not args.no_api:
    try:
      api = api_rate(wl, args.envs or wl.n_envs, local_rank, args.steps)
    except Exception as ex:   # reported, never silently dropped
      api = dict(error='%s: %s' % (type(ex).__name__, ex))
    torch.cuda.empty_cache()

  sampler = ClockSampler(local_rank) if rank == 0 else None
  b = Bench(wl, args, world, rank, local_rank, args.steps, args.warmup, E=args.envs or None)
  res = b.run(sampler, args.dump_outputs if rank == 0 else None)
  clocks = sampler.stop() if sampler else None
  e2e = None if args.no_e2e else b.e2e()
  collective = ('none' if world == 1 else
                'frames stored into every rank\'s gathered buffer by the render kernel '
                '(NVLink peer memory) + one NCCL all-gather of the 11-byte per-env records (reward, step type, '
                'success, status), which is also the completion barrier'
                if b.peer is not None and b.gather == 'peer' else
                'render into the rank\'s block of the gathered buffer, copy-engine pushes to '
                'the peers over NVLink + one-element NCCL all-reduce as completion barrier'
                if b.peer is not None else
                'NCCL all_gather of frames per step (async, overlaps the next step)')
  cfg = workload_config(wl, b.E)
  cfg.update(auto_reset='pooled scenes', pool_depth=b.K, collective=collective,
             l2='frame ring of %d buffers (%.0f MB) > L2, no flush'
             % (b.n_ring, b.n_ring * b.frame_bytes / 1e6),
             headline='BASELINE.json configs[1] (the config the metric is quoted on); the other '
                      'configs are under "configs", measured in the same run')
  if numa is not None:
    cfg['numa_node'] = numa
  traffic, traffic_src = _traffic(args.workload)
  roof = b.roofline(res['render_ms'], traffic)
  if traffic_src:
    roof['traffic_source'] = traffic_src
  headline_E = b.E
  b.close()

  # ---- the variant without the episode-length reset (SURVEY 8d asks for both) ---------------
  extra = {}
  if world == 1 and args.also != 'none':
    bi = Bench(wl, args, world, rank, local_rank, min(args.steps, 100), 5, E=args.envs or None,
               max_episode_length=2 ** 31 - 1)
    r = bi.run()
    extra['max_episode_length_inf'] = dict(
        value=r['value'], unit=UNIT, ms_per_step=r['ms_per_step'],
        note='max_episode_length = 2^31-1: envs reset only when the task terminates them')
    bi.close()

  # ---- the other BASELINE configs, same run ----------------------------------------------------
  also = args.also
  if also is None:
    also = 'c3,c4,c5' if world == 1 else 'c4,c5'
  configs = {}
  for key in [k for k in also.split(',') if k and k != 'none' and k != args.workload]:
    w2 = workloads.WORKLOADS[key]()
    b2 = Bench(w2, args, world, rank, local_rank, min(args.steps, 100), 5)
    r2 = b2.run()
    t2, _ = _traffic(key)
    entry = dict(value=r2['value'], unit=UNIT, ms_per_step=r2['ms_per_step'], n_gpus=world,
                 config=workload_config(w2, b2.E), timed=r2['timed'],
                 roofline=b2.roofline(r2['render_ms'], t2), gpu_launches=r2['launches'])
    for k in ('frames_sharded', 'nvlink'):
      if k in r2:
        entry[k] = r2[k]
    if world == 1 and key in ('c4', 'c5'):
      entry['note'] = 'per-GPU shard of the 8-GPU config (envs_per_gpu of the full batch / 8)'
    configs[key] = entry
    b2.close()

  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return

  cpu = None
  if not args.no_cpu_baseline and world == 1:
    n_cpu_steps = 25
    v, cores, dt, n = cpu_reference(wl, 512 * usable_cores(), n_cpu_steps, 3)
    v1 = cpu_reference(wl, 32, 10, 2, cores=1)[0]
    cpu = dict(value=v, unit=UNIT, cores=cores, kind='port', single_core=v1,
               sample='%d envs x %d steps of %s, %.1f s wall, oracle C port of the reference '
                      'path (Pillow polygon fill + LANCZOS restated), one thread per usable core '
                      '(affinity mask capped by the cgroup CPU quota; %d logical CPUs visible)'
                      % (n, n_cpu_steps, wl.name, dt, os.cpu_count() or 1))
    cpu.update(pillow_check())
  line = dict(
      metric=METRIC, value=res['value'], unit=UNIT, frames_per_sec=res['value'], n_gpus=world,
      steps=args.steps, warmup=args.warmup, ms_per_step=res['ms_per_step'], higher_is_better=True,
      scaling='weak', vs_baseline=None, dtype='u8', data='synthetic', config=cfg, timed=res['timed'],
      roofline=roof, cpu_baseline=cpu, e2e=e2e, gpu_launches=res['launches'], clocks=clocks)
  for k in ('frames_sharded', 'nvlink'):
    if k in res:
      line[k] = res[k]
  line.update(extra)
  if configs:
    line['configs'] = configs
  if api is not None:
    line['api'] = api
  print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def pillow_check():
  """If Pillow is importable on this box: the real ImageDraw.polygon + resize(LANCZOS) per
  frame of the headline workload's geometry, on one core -- so that the port's rate can be
  read against the library the reference calls (BASELINE.md section 3)."""
  try:
    from PIL import Image, ImageDraw
  except Exception:
    return dict(pillow_ms_per_frame=None)
  rng = np.random.RandomState(3)
  n, S, aa, size = 200, 5, 5, 64
  cs = size * aa
  polys = []
  for _ in range(n * S):
    cx, cy = rng.uniform(0.1, 0.9, 2) * cs
    r = 0.13 * cs * 0.6
    k = rng.choice([3, 4, 24])
    ang = np.linspace(0, 2 * np.pi, k, endpoint=False)
    polys.append([(float(cx + r * np.cos(a)), float(cy + r * np.sin(a))) for a in ang])
  lanczos = getattr(Image, 'LANCZOS', None) or Image.Resampling.LANCZOS
  t0 = time.perf_counter()
  for i in range(n):
    canvas = Image.new('RGB', (cs, cs), (0, 0, 0))
    draw = ImageDraw.Draw(canvas)
    for p in polys[i * S:(i + 1) * S]:
      draw.polygon(p, fill=(200, 100, 50))
    np.flipud(np.array(canvas.resize((size, size), lanczos)))
  ms = 1e3 * (time.perf_counter() - t0) / n
  return dict(pillow_ms_per_frame=ms, pillow_frames_per_sec_per_core=1e3 / ms,
              pillow_note='PIL %s: Image.new + %d ImageDraw.polygon + resize(LANCZOS) + flipud per '
                          '64x64 aa=5 frame, one core, no env logic' % (
                              getattr(__import__('PIL'), '__version__', '?'), S))


if __name__ == '__main__':
  main()
