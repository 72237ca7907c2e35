#!/usr/bin/env python
"""Benchmark: env-steps/s of the batched Melting Pot hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 2|3|4|5] [--gather-obs]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path (state transition + all observations rendered) over one batch of env
instances per GPU under uniform-random actions. --config picks the BASELINE.json configuration:
  2 (default, the headline)  clean_up, 7 players, 4096 envs per GPU
  3                          commons_harvest__open, 16 players, 8192 envs per GPU
  4                          territory__rooms, 9 players, 2048 envs per GPU (16384 over 8 GPUs)
  5                          the 8-substrate sweep, 2048 envs each, substrates dealt round-robin over the ranks
Fields of the JSON line:
  value     device-resident throughput: actions already in HBM, outputs left in HBM.
  e2e       the same metric through the host-buffer C-ABI calls (pinned host actions in, EVERY observation copied
            back to pinned host memory each step), pipelined over two buffer sets (mp_step_host_async / mp_wait).
  roofline  the render kernel's achieved HBM bandwidth (algorithmic bytes / CUDA-event time of its launches).
  cpu_baseline  the C oracle (a port of the reference semantics; DMLab2D itself cannot run here), N = 1 only.
Under torchrun (N > 1) every rank steps its own shard of envs; the stacked timestep (reward / discount / step type of
every env of every rank) reaches every rank through peer-memory stores fused into the state-transition kernel
(mp_exchange_*), and after the timed region every rank replays a few envs of its neighbour's shard and compares them
with what it received ("shard_check").
"""

import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

_ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, _ROOT)

METRIC = 'env_steps_per_sec'
UNIT = 'env-steps/s'

SWEEP = [('clean_up', 7), ('commons_harvest__open', 7), ('commons_harvest__closed', 7), ('commons_harvest__partnership', 7),
         ('territory__rooms', 9), ('territory__open', 9), ('territory__inside_out', 5), ('coins', 2)]
CONFIGS = {
    2: dict(jobs=[('clean_up', 7)], envs=4096, label='BASELINE.json configs[1]: clean_up, 7 players, 4096 batched envs per GPU'),
    3: dict(jobs=[('commons_harvest__open', 16)], envs=8192,
            label='BASELINE.json configs[2]: commons_harvest__open, 16 players, 8192 envs per GPU'),
    4: dict(jobs=[('territory__rooms', 9)], envs=2048,
            label='BASELINE.json configs[3]: territory__rooms, 9 players, 2048 envs per GPU (16384 sharded over 8)'),
    5: dict(jobs=SWEEP, envs=2048, label='BASELINE.json configs[4]: 8-substrate sweep x 2048 envs each, substrates dealt over the ranks'),
}


def _peaks():
  path = os.path.join(_ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
  return 6650.0, 'fallback (B200_PROFILING.md)'


def _render_source_hash():
  h = hashlib.sha1()
  for name in ('render.cuh', 'common.cuh'):
    with open(os.path.join(_ROOT, 'meltingpot_b200', 'csrc', name), 'rb') as f:
      h.update(f.read())
  return h.hexdigest()


def _traffic_per_launch(substrate, players, num_envs):
  """dram bytes per render launch from the committed `ncu --set full` capture of THIS kernel source, scaled to the
  batch; None when no capture of the current render.cuh / common.cuh exists for the substrate (a stale number is
  worse than none)."""
  path = os.path.join(_ROOT, 'profiles', 'render_traffic.json')
  if not os.path.exists(path):
    return None
  with open(path) as f:
    rec = json.load(f)
  ent = rec.get('captures', {}).get(f'{substrate}__{players}p')
  if not ent or ent.get('source_sha1') != _render_source_hash():
    return None
  return ent['dram_bytes_per_env'] * num_envs


class ClockSampler(threading.Thread):
  """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

  QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
           'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
           'clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index = index
    self.samples = []
    self._halt = threading.Event()

  def run(self):
    while not self._halt.is_set():
      try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                              '-i', str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
          self.samples.append([s.strip() for s in out.split(',')])
      except Exception:  # pylint: disable=broad-except
        pass
      self._halt.wait(0.05)

  def stop(self):
    self._halt.set()
    self.join(timeout=5)
    if not self.samples:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
    sm = [float(s[0]) for s in self.samples if s[0].replace('.', '').isdigit()]
    mx = [float(s[1]) for s in self.samples if s[1].replace('.', '').isdigit()]
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    reasons = [n for i, n in enumerate(names) if any(s[2 + i] == 'Active' for s in self.samples if len(s) > 2 + i)]
    return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': reasons, 'samples': len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# NUMA: a rank's pinned host buffers must live on the node its GPU hangs off, or the device->host stream crosses the
# socket interconnect (GPU0-3 -> node 0, GPU4-7 -> node 1 on the 8-GPU boxes).
# ---------------------------------------------------------------------------------------------------------------------
def gpu_selector(local_rank):
  """What `nvidia-smi -i` should be given for CUDA device `local_rank`: its UUID when torch reports one (an index would
  name the wrong GPU under CUDA_VISIBLE_DEVICES), else the index."""
  try:
    import torch
    uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    if uuid and uuid != 'None':
      return uuid if uuid.startswith('GPU-') else 'GPU-' + uuid
  except Exception:  # pylint: disable=broad-except
    pass
  return str(local_rank)


def bind_to_gpu_numa_node(local_rank):
  """Pins this process (CPU affinity + preferred memory node) to the NUMA node of GPU `local_rank`. Best effort."""
  info = {'node': None, 'cpus': None, 'mempolicy': False}
  try:
    bus = subprocess.run(['nvidia-smi', '--query-gpu=pci.bus_id', '--format=csv,noheader', '-i', gpu_selector(local_rank)],
                         capture_output=True, text=True, timeout=10).stdout.strip().lower()
    if bus.startswith('00000000:'):
      bus = bus[4:]  # sysfs uses a 4-digit PCI domain
    with open(f'/sys/bus/pci/devices/{bus}/numa_node') as f:
      node = int(f.read().strip())
    if node < 0:
      return info
    with open(f'/sys/devices/system/node/node{node}/cpulist') as f:
      cpus = set()
      for part in f.read().strip().split(','):
        lo, _, hi = part.partition('-')
        cpus.update(range(int(lo), int(hi or lo) + 1))
    allowed = cpus & os.sched_getaffinity(0)
    if allowed:
      os.sched_setaffinity(0, allowed)
    info.update(node=node, cpus=len(allowed))
    # set_mempolicy(MPOL_PREFERRED = 1, nodemask) -- syscall 238 on x86-64
    mask = ctypes.c_ulong(1 << node)
    libc = ctypes.CDLL(None, use_errno=True)
    if libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(64)) == 0:
      info['mempolicy'] = True
  except Exception:  # pylint: disable=broad-except
    pass
  return info


def _load_blob(name, players):
  from meltingpot_b200 import substrates
  return substrates.load_blob(name, ('default',) * players)


def _oracle_rate(blob, cores, seconds):
  """Env-steps/s of the oracle on `cores` threads, one persistent env per thread, full rendering; >= `seconds` of work."""
  from oracle import binding as oracle_binding
  oracle_binding.build()
  batch = oracle_binding.OracleBatch(blob, cores, seed=1)
  t0 = time.perf_counter()
  n = batch.step_random(50, cores)
  rate = n / (time.perf_counter() - t0)
  steps = max(50, int(rate * seconds / cores))
  t0 = time.perf_counter()
  n = batch.step_random(steps, cores)
  dt = time.perf_counter() - t0
  batch.close()
  return n / dt, steps, dt


def cpu_baseline(jobs, seconds=12.0):
  """Times the oracle on all host cores over a bounded sample of the same workload; returns the cpu_baseline object."""
  cores = os.cpu_count() or 1
  total_n, total_t, parts = 0.0, 0.0, []
  for name, players in jobs:
    rate, steps, dt = _oracle_rate(_load_blob(name, players), cores, seconds / len(jobs))
    total_n += rate * dt
    total_t += dt
    parts.append(f'{name} {players}p: {cores} envs x {steps} steps')
  return {'value': total_n / total_t, 'unit': UNIT, 'cores': cores, 'kind': 'port',
          'sample': '; '.join(parts) + f'; one persistent env per thread, uniform-random actions, every player RGB + WORLD.RGB '
                                       f'rendered each step, {total_t:.1f} s of wall time'}


def run_reference(args, rank, world):
  """--impl reference: the CPU implementation of the path (oracle port) on all host cores, same config."""
  if rank != 0:
    return
  from oracle import binding as oracle_binding
  oracle_binding.build()
  cfg = CONFIGS[args.config]
  cores = os.cpu_count() or 1
  blobs = [(name, players, _load_blob(name, players)) for name, players in cfg['jobs']]
  batches = [(name, players, oracle_binding.OracleBatch(blob, cores, seed=1)) for name, players, blob in blobs]
  # A bench "step" of this arm is a bounded sample: `per_step` env-steps on each of `cores` persistent envs (per
  # substrate of the config). Sized from a short calibration so that the K timed steps take about `--ref-seconds`.
  t0 = time.perf_counter()
  n = sum(b.step_random(8, cores) for _, _, b in batches)
  rate = n / (time.perf_counter() - t0)
  per_step = max(8, int(rate * args.ref_seconds / max(args.steps, 1) / (cores * len(batches))))
  for _ in range(args.warmup):
    for _, _, b in batches:
      b.step_random(per_step, cores)
  t0 = time.perf_counter()
  total = 0
  for _ in range(args.steps):
    for _, _, b in batches:
      total += b.step_random(per_step, cores)
  dt = time.perf_counter() - t0
  for _, _, b in batches:
    b.close()
  value = total / dt
  sample = (f'{cores} persistent envs per substrate (one per thread) x {per_step} env-steps per bench step, {args.steps} steps, '
            f'{dt:.1f} s, full rendering of every observation each env-step')
  line = {
      'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / max(args.steps, 1) * 1e3,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
      'config': {'workload': cfg['label'] + '; CPU oracle port of the reference path on the host cores (DMLab2D itself is not '
                             'installable here), bounded sample of the same substrates / player counts',
                 'bench_config': args.config, 'envs': cores * len(batches)},
      'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
      'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'agent_steps_per_sec': value * sum(p for _, p in cfg['jobs']) / len(cfg['jobs']),
  }
  _emit(line)


class Job:
  """One substrate on this rank: engine, action stream and (N > 1) the timestep exchange."""

  def __init__(self, name, players, B, rank, world, local_rank, steps, warmup, exchange):
    import torch
    from meltingpot_b200 import engine
    self.name, self.B, self.rank, self.world = name, B, rank, world
    self.blob = _load_blob(name, players)
    self.eng = engine.Engine(self.blob, B, device=local_rank, seed=1, env_index_base=rank * B)
    self.P, self.A = self.eng.num_players, self.eng.num_actions
    self.dev = torch.device('cuda', local_rank)
    self.n_actions = steps + warmup
    self.actions = self.make_actions(rank)
    self.stream = torch.cuda.current_stream(self.dev)
    self.side = None
    self.exchange = exchange and world > 1
    if self.exchange:
      from meltingpot_b200 import distributed
      distributed.connect_exchange(self.eng)
      self.side = torch.cuda.Stream(device=self.dev)
      self.stepped = torch.cuda.Event()

  def make_actions(self, owner_rank):
    import torch
    gen = torch.Generator(device=self.dev).manual_seed(1234 + owner_rank)
    return torch.randint(0, self.A, (self.n_actions, self.B, self.P), generator=gen, device=self.dev, dtype=torch.int32)

  def reset(self):
    self.eng.reset()

  def step(self, t):
    if not self.exchange:
      self.eng.step(self.actions[t])
      return
    # The state-transition kernel writes this rank's packed timestep rows into every rank's gathered buffer (peer
    # stores over NVLink) as it produces them; the two kernels of the step stay back to back on the main stream (the
    # renderer's prologue overlaps the transition's tail). The consumer-side wait for the other ranks' rows is a
    # one-warp kernel on a side stream, off the critical path.
    self.eng.step(self.actions[t])
    self.stepped.record(self.stream)
    self.side.wait_event(self.stepped)
    self.eng.exchange_wait(self.side)

  def join(self):
    if self.side is not None:
      self.stream.wait_stream(self.side)


def shard_check(job, n_check=8):
  """Outside the timed region: this rank replays the first `n_check` envs of its right neighbour's shard from the
  same seed and actions on a fresh engine and compares (i) the rows it RECEIVED through the exchange for the last
  step and (ii) the neighbour's final avatar state / sprite grid / WORLD.RGB (all-gathered for the check) with its own
  replay. Any sharding mistake (seed base, action slice, row placement in the gathered buffer) fails it."""
  import torch
  import torch.distributed as dist
  from meltingpot_b200 import engine
  eng, B, P, world, rank = job.eng, job.B, job.P, job.world, job.rank
  nb = (rank + 1) % world
  torch.cuda.synchronize()
  received = eng.gathered_timestep()[nb * B: nb * B + n_check].clone()
  mine = torch.cat([eng.avatar_state[:n_check].reshape(n_check, -1).to(torch.int64),
                    eng.grid[:n_check].reshape(n_check, -1).to(torch.int64),
                    eng.world_rgb[:n_check].reshape(n_check, -1).to(torch.int64)], dim=1).contiguous()
  everyone = torch.empty((world,) + tuple(mine.shape), dtype=mine.dtype, device=mine.device)
  dist.all_gather_into_tensor(everyone, mine)
  replay = engine.Engine(job.blob, n_check, device=eng.device, seed=1, env_index_base=nb * B)
  acts = job.make_actions(nb)[:, :n_check].contiguous()
  replay.reset()
  for t in range(job.n_actions):
    replay.step(acts[t])
  torch.cuda.synchronize()
  want = torch.cat([replay.avatar_state.reshape(n_check, -1).to(torch.int64), replay.grid.reshape(n_check, -1).to(torch.int64),
                    replay.world_rgb.reshape(n_check, -1).to(torch.int64)], dim=1)
  ok_state = bool((everyone[nb] == want).all())
  ok_rows = bool((received == replay.timestep_packed).all())
  replay.close()
  flag = torch.tensor([1 if (ok_state and ok_rows) else 0], device=mine.device)
  dist.all_reduce(flag, op=dist.ReduceOp.MIN)
  if int(flag.item()) == 1:
    return 'ok'
  return f'MISMATCH (rank {rank}: state {ok_state}, received rows {ok_rows})'


def time_job(job, K, Wm, dist, sampler=None):
  """W warm-up steps, then exactly K timed steps bracketed by barrier + synchronize; returns (elapsed_ms, launches)."""
  import torch
  job.reset()
  for t in range(Wm):
    job.step(t)
  job.join()
  torch.cuda.synchronize()
  if sampler is not None:
    sampler.start()
  if dist is not None:
    dist.barrier()
  torch.cuda.synchronize()
  launches0 = job.eng.launch_count()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record(job.stream)
  for t in range(Wm, Wm + K):
    job.step(t)
  job.join()
  ev1.record(job.stream)
  torch.cuda.synchronize()
  if dist is not None:
    dist.barrier()
  return ev0.elapsed_time(ev1), job.eng.launch_count() - launches0


DUMP_ENVS = 16            # env instances per run whose images --dump-outputs writes (a whole batch's run to gigabytes)
DUMP_LIMIT = 64 << 20     # bytes --dump-outputs may write in one run, over all ranks and substrates


def dump_outputs(job, out_dir, prefix, n_envs, budget):
  """Writes what the last timed step handed its caller as `out_dir/<prefix><name>.npy` (float32 images, float64 else):
  reward, discount, step_type, scalar_obs and event_count of every env, and rgb, world_rgb and events (unused slots
  zeroed) of a fixed, seeded sample of `n_envs` envs, whose indices are `sample_envs`. Writes nothing and exits if
  that is more than `budget` bytes; returns the bytes written."""
  import numpy as np
  import torch
  eng = job.eng
  idx = np.sort(np.random.default_rng(0).choice(job.B, size=min(n_envs, job.B), replace=False))
  sel = torch.as_tensor(idx, device=job.dev)
  events = eng.events[sel].cpu().numpy()
  used = np.arange(events.shape[1])[None, :] < eng.event_count[sel].cpu().numpy()[:, None]
  arrays = {
      'reward': eng.reward.cpu().numpy(), 'discount': eng.discount.cpu().numpy(),
      'step_type': eng.step_type.cpu().numpy().astype(np.float64),
      'scalar_obs': eng.scalar_obs[:eng.num_scalar_obs].cpu().numpy(),
      'event_count': eng.event_count.cpu().numpy().astype(np.float64),
      'sample_envs': idx.astype(np.float64),
      'rgb': eng.rgb[sel].cpu().numpy().astype(np.float32),
      'world_rgb': eng.world_rgb[sel].cpu().numpy().astype(np.float32),
      'events': np.where(used[..., None], events, 0).astype(np.float64),
  }
  total = sum(a.nbytes for a in arrays.values())
  if total > budget:
    raise SystemExit(f'bench.py: --dump-outputs would write {total} bytes for {prefix[:-1]}, over the {budget} left of the '
                     f'{DUMP_LIMIT} bytes a run may write')
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, f'{prefix}{name}.npy'), a)
  return total


def render_roofline(job, K, Wm):
  """The render kernel alone: CUDA events around each launch on the launching stream."""
  import torch
  n_r = min(K, 50)
  evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_r)]
  for i in range(n_r):
    job.eng.step_state(job.actions[Wm + i])
    evs[i][0].record(job.stream)
    job.eng.render()
    evs[i][1].record(job.stream)
  torch.cuda.synchronize()
  return statistics.mean(a.elapsed_time(b) for a, b in evs)


def measure_pcie_d2h(dev, nbytes=1 << 30):
  """Plain pinned device->host copy rate on this rank's link (what bounds the e2e path)."""
  import torch
  src = torch.empty(nbytes, dtype=torch.uint8, device=dev)
  dst = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
  dst.copy_(src, non_blocking=True)
  torch.cuda.synchronize()
  best = 0.0
  for _ in range(3):
    t0 = time.perf_counter()
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    best = max(best, nbytes / (time.perf_counter() - t0) / 1e9)
  return best


def run_e2e(job, n_e, dist, images=True):
  """End to end through the C ABI with HOST buffers, pipelined over two buffer sets: while step t's observations cross
  PCIe into set t & 1, step t + 1's kernels already run. The consumer touches every returned reward (a host read of
  the step's result) after mp_wait. Returns (seconds, h2d bytes, d2h bytes per step)."""
  import torch
  eng = job.eng
  outs = [eng.make_host_outputs(rgb=images, world_rgb=images) for _ in range(2)]
  for o in outs:
    o.pop('events', None)
  host_actions = job.actions[:n_e + 2].cpu().pin_memory()
  d2h = sum(t.numel() * t.element_size() for k, t in outs[0].items() if k in ('rgb', 'world_rgb', 'scalar_block'))
  h2d = host_actions[0].numel() * host_actions[0].element_size()
  for i in range(2):  # warm-up: allocates the second device image set, pages in the pinned buffers
    eng.step_host_async(host_actions[i], outs[i], i)
  eng.wait(0); eng.wait(1)
  torch.cuda.synchronize()
  if dist is not None:
    dist.barrier()
  checksum = 0.0
  t0 = time.perf_counter()
  for i in range(n_e):
    slot = i & 1
    if i >= 2:
      eng.wait(slot)
      checksum += float(outs[slot]['reward'].sum())
    eng.step_host_async(host_actions[2 + i], outs[slot], slot)
  for i in range(max(0, n_e - 2), n_e):
    eng.wait(i & 1)
    checksum += float(outs[i & 1]['reward'].sum())
  dt = time.perf_counter() - t0
  return dt, h2d, d2h, checksum


def run_gather_obs(job, n_g, dist, world, rank):
  """Steps with the renderer also delivering every strip into every rank's stacked observation buffer (mp_gather_obs_*,
  TMA bulk stores over NVLink peer mappings). Returns (ms per step, bytes each rank sends to its peers per step)."""
  import torch
  eng = job.eng
  if world > 1:
    from meltingpot_b200 import distributed
    distributed.connect_gather_obs(eng)
  else:
    ptr, _ = eng.gather_obs_create(0, 1)
    eng.gather_obs_connect([ptr])
  for t in range(3):
    job.step(t)
  job.join()
  eng.gather_obs_wait()
  torch.cuda.synchronize()
  if dist is not None:
    dist.barrier()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record(job.stream)
  for t in range(n_g):
    job.step(3 + t)
  job.join()
  eng.gather_obs_wait()  # the consumer-side wait for every rank's last delivery closes the timed region
  ev1.record(job.stream)
  torch.cuda.synchronize()
  if dist is not None:
    dist.barrier()
  ms = ev0.elapsed_time(ev1) / n_g
  ok = None
  if world > 1:  # what arrived from the right neighbour equals what it holds (checked through an NCCL all-gather of hashes)
    rgb, wrgb = eng.gathered_observations()
    B = job.B
    mine = torch.stack([eng.rgb.to(torch.int64).sum(), eng.world_rgb.to(torch.int64).sum()])
    every = torch.empty((world, 2), dtype=torch.int64, device=mine.device)
    dist.all_gather_into_tensor(every, mine)
    got = torch.stack([torch.stack([rgb[r * B:(r + 1) * B].to(torch.int64).sum(), wrgb[r * B:(r + 1) * B].to(torch.int64).sum()]) for r in range(world)])
    flag = torch.tensor([1 if bool((got == every).all()) else 0], device=mine.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = 'ok' if int(flag.item()) == 1 else 'MISMATCH'
  eng.gather_obs_enable(False)
  obs_bytes = eng.rgb.numel() + eng.world_rgb.numel()
  return ms, obs_bytes * max(world - 1, 0), obs_bytes, ok


def run_b200(args, rank, world, local_rank):
  import torch
  if not torch.cuda.is_available():
    raise SystemExit('bench.py: no CUDA device; the B200 engine has no CPU path')
  numa = bind_to_gpu_numa_node(local_rank)  # before any pinned allocation (first touch decides the node)
  torch.cuda.set_device(local_rank)
  dist = None
  if world > 1:
    import torch.distributed as dist  # pylint: disable=g-import-not-at-top
    dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
  cfg = CONFIGS[args.config]
  B = args.envs or cfg['envs']
  K, Wm = args.steps, args.warmup
  dev = torch.device('cuda', local_rank)
  my_jobs = [j for i, j in enumerate(cfg['jobs']) if i % world == rank] if len(cfg['jobs']) > 1 else list(cfg['jobs'])
  single = len(cfg['jobs']) == 1
  peak, peak_src = _peaks()

  def max_over_ranks(x):
    if world == 1:
      return x
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  sampler = ClockSampler(gpu_selector(local_rank)) if rank == 0 else None
  per_job, elapsed_ms, launches, env_steps = [], 0.0, 0, 0
  dumped = 0
  shard = None
  e2e = e2e_scalars = gather = None
  first_job = None
  for ji, (name, players) in enumerate(my_jobs):
    job = Job(name, players, B, rank, world, local_rank, K, Wm, exchange=single)
    ms, n_l = time_job(job, K, Wm, dist if single else None, sampler if ji == 0 else None)
    if ji == 0 and sampler is not None:
      clocks = sampler.stop()
    if args.dump_outputs:  # before anything below steps the engine again; each rank keeps to its share of the limit
      prefix = (f'rank{rank}.' if world > 1 else '') + f'{name}.'
      dumped += dump_outputs(job, args.dump_outputs, prefix, max(1, DUMP_ENVS // (world * len(my_jobs))),
                             DUMP_LIMIT // world - dumped)
    elapsed_ms += ms
    launches += n_l
    env_steps += B * K
    algo_bytes, render_bytes = job.eng.algorithmic_bytes()
    if single and world > 1:
      shard = shard_check(job)
    render_ms = render_roofline(job, K, Wm)
    achieved = render_bytes * B / (render_ms * 1e-3) / 1e9
    per_job.append({'substrate': name, 'players': job.P, 'envs': B, 'ms_per_step': ms / K, 'env_steps_per_sec': B * K / (ms * 1e-3),
                    'render_ms': render_ms, 'render_gbs': achieved, 'render_frac': achieved / peak,
                    'whole_step_frac': algo_bytes * B * K / (ms * 1e-3) / 1e9 / peak, 'layout': job.eng.render_plan()})
    if ji == 0:
      first_job = dict(name=name, players=job.P, algo_bytes=algo_bytes, render_bytes=render_bytes, render_ms=render_ms, achieved=achieved)
      if single:
        # ---- end to end through the host-buffer C-ABI calls --------------------------------------------
        n_e = max(4, min(K, args.e2e_steps))
        dt, h2d, d2h, _ = run_e2e(job, n_e, dist, images=True)
        dt = max_over_ranks(dt)
        pcie = measure_pcie_d2h(dev)
        e2e = {'value': world * B * n_e / dt, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'steps': n_e,
               'api': 'mp_step_host_async + mp_wait (C ABI, pinned host buffers, two buffer sets; every observation copied back, '
                      'scalars as one packed block)',
               'pcie_d2h_gbs_measured_rank0': pcie, 'frac_of_pcie': (d2h * n_e / dt / 1e9) / pcie if pcie else None, 'numa': numa}
        n_s = max(n_e, min(K, 200))
        dt_s, h2d_s, d2h_s, _ = run_e2e(job, n_s, dist, images=False)
        dt_s = max_over_ranks(dt_s)
        e2e_scalars = {'value': world * B * n_s / dt_s, 'unit': UNIT, 'h2d_bytes_per_step': h2d_s, 'd2h_bytes_per_step': d2h_s,
                       'steps': n_s, 'api': 'same calls with NULL image pointers (images stay in HBM for a GPU-resident consumer)'}
        if args.gather_obs:
          n_g = max(4, min(K, 24))
          ms_g, sent, obs_bytes, ok = run_gather_obs(job, n_g, dist, world, rank)
          ms_g = max_over_ranks(ms_g)
          gather = {'value': world * B / (ms_g * 1e-3), 'unit': UNIT, 'ms_per_step': ms_g, 'steps': n_g,
                    'obs_bytes_per_rank_per_step': obs_bytes, 'nvlink_bytes_sent_per_rank_per_step': sent,
                    'nvlink_gbs_per_gpu_egress': sent / (ms_g * 1e-3) / 1e9, 'nvlink_peak_gbs_per_direction': 900.0,
                    'frac_of_nvlink': sent / (ms_g * 1e-3) / 1e9 / 900.0, 'check': ok,
                    'how': 'k_render<GATHER> hands every finished strip to one TMA bulk store per rank (peer memory over NVLink / NVSwitch) '
                           'next to the local one; two stacked buffers per rank (slot = step parity), flag wait kernel on the consumer side'}
    job.eng.close()
    del job
  if not single and dist is not None:
    dist.barrier()
  elapsed_ms = max_over_ranks(elapsed_ms)
  if world > 1:
    tot = torch.tensor([float(env_steps), float(launches)], dtype=torch.float64, device=dev)
    dist.all_reduce(tot)
    env_steps_all, launches_all = float(tot[0].item()), int(tot[1].item())
    gathered_jobs = [None] * world
    dist.all_gather_object(gathered_jobs, per_job)
    per_job_all = [j for r in gathered_jobs for j in r]
  else:
    env_steps_all, launches_all, per_job_all = float(env_steps), launches, per_job
  value = env_steps_all / (elapsed_ms * 1e-3)

  if rank == 0:
    fj = first_job
    if single:
      multi = ('env shards, no data-path collective; the stacked reward/discount/step_type rows reach every rank by peer-memory stores '
               'issued by the state-transition kernel itself (NVLink, mp_exchange_*), consumer-side flag wait on a side stream') if world > 1 else 'single GPU'
    else:
      multi = f'substrates dealt round-robin over {world} rank(s); independent jobs, no exchange; per-rank time = sum over its substrates'
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': Wm,
        'ms_per_step': elapsed_ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'u8', 'data': 'synthetic',
        'config': {
            'workload': cfg['label'] + ', uniform-random actions, WORLD.RGB on',
            'bench_config': args.config, 'envs_per_gpu': B, 'players': fj['players'] if single else [p for _, p in cfg['jobs']],
            'global_envs': world * B if single else B * len(cfg['jobs']),
            'cache': 'per-step working set (freshly written observations, >= 0.4 GB) >> 126 MB L2; no explicit flush',
            'multi_gpu': multi,
        },
        'agent_steps_per_sec': sum(j['env_steps_per_sec'] * j['players'] for j in per_job_all) if not single else value * fj['players'],
        'gpu_launches': launches_all,
        'clocks': clocks,
        'roofline': {'bound': 'hbm', 'kernel': 'k_render', 'substrate': fj['name'], 'achieved': fj['achieved'], 'peak': peak, 'unit': 'GB/s',
                     'frac': fj['achieved'] / peak, 'traffic': _traffic_per_launch(fj['name'], fj['players'], B), 'peak_source': peak_src,
                     'algorithmic_bytes_per_launch': fj['render_bytes'] * B, 'ms_per_launch': fj['render_ms'],
                     'whole_step_algorithmic_bytes_per_env': fj['algo_bytes'],
                     'whole_step_frac': per_job_all[0]['whole_step_frac'] if single else None},
        'per_substrate': per_job_all,
    }
    if e2e is not None:
      line['e2e'] = e2e
      line['e2e_scalars_only'] = e2e_scalars
    if shard is not None:
      line['shard_check'] = shard
    if gather is not None:
      line['gather_obs'] = gather
    if not args.no_cpu_baseline and world == 1:
      line['cpu_baseline'] = cpu_baseline(cfg['jobs'], seconds=args.ref_seconds)
    _emit(line)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


_STDOUT_FD = []  # the real stdout, saved by main() while fd 1 points at stderr


def _emit(line):
  sys.stdout.flush()
  if _STDOUT_FD:
    os.dup2(_STDOUT_FD[0], 1)
  print(json.dumps(line), flush=True)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=2000)
  ap.add_argument('--warmup', type=int, default=20)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--config', type=int, default=2, choices=sorted(CONFIGS))
  ap.add_argument('--envs', type=int, default=0, help='env instances per GPU (default: the config\'s)')
  ap.add_argument('--e2e-steps', type=int, default=40)
  ap.add_argument('--ref-seconds', type=float, default=15.0, help='CPU arm / cpu_baseline: seconds of oracle work to time')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--gather-obs', action='store_true', help='also measure steps with the stacked-observation gather over NVLink')
  ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<substrate>.<name>.npy, '
                                                        'at most 64 MB per run (seeded inputs: two builds can be compared '
                                                        'output for output; --impl b200 only)')
  args = ap.parse_args()
  if args.dump_outputs and args.impl != 'b200':
    ap.error('--dump-outputs writes the outputs of the b200 path; --impl reference computes none to compare')
  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  # Exactly one JSON line on stdout: native libraries (NCCL prints its version banner there) write to the stdout
  # file descriptor, so everything but the final line is sent to stderr.
  sys.stdout.flush()
  _STDOUT_FD.append(os.dup(1))
  os.dup2(2, 1)
  if args.impl == 'reference':
    run_reference(args, rank, world)
  else:
    run_b200(args, rank, world, local_rank)


if __name__ == '__main__':
  main()
