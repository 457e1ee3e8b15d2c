#!/usr/bin/env python
"""Benchmark of the GP-Bandit suggest() hot path (BASELINE.json metric).

metric   : GP-UCB candidates scored/sec; suggest() latency at N=1000, D=20, M=100k pool
workload : c2 (default) -- GP posterior mu/var + UCB (+trust region) over M=100k candidates per GPU,
           N=1000 trials, D=20, fp64 (weak scaling: every rank scores its own M-candidate shard of one
           global Philox pool, then ONE fused NVLink exchange+merge kernel picks the global arg-max).
           c5 (--workload c5) -- M=1M candidates split over the ranks, N=2000, D=50 (BASELINE C5).
step     : one pass of the fused scoring kernel over the rank's candidates + device top-1 + the exchange.
value    : candidates/s with candidates resident in HBM (CUDA events on the launching stream, max over
           ranks); per-step event times of every rank are reported (min / median / max) so that a stall
           is attributable.
e2e      : the same step through ONE C-ABI call with HOST buffers (`vzgp_suggest_host`): H2D of the M x D
           candidates, scoring, top-1, exchange+merge across ranks, D2H of all M scores and the winner,
           host-synchronous - inside the timed region, at every N.
suggest_e2e (N=1): wall-clock of a whole `VizierGPBandit.suggest(1)` (trial conversion + 4x50 ARD + fit +
           acquisition optimisation) on 1000 completed 20-D trials after one new trial arrives, with the
           M=100k random-pool optimiser (the metric's configuration) and with the default Eagle optimiser,
           next to the same pipeline restated on the CPU (NumPy/SciPy oracle, all host cores).
roofline : the scoring kernel is FP64-pipe bound (N^2 flops per candidate against 8(D+1) bytes), so
           `achieved` is algorithmic TFLOP/s against the FP64 DMMA peak measured on this pool's B200 by
           tools/fp64_peak.cu (profiles/fp64_peak_r01.json; MEASURED_PEAKS.json has no fp64 entry); the
           HBM view is reported beside it.
cpu_baseline / --impl reference: the NumPy/SciPy oracle (a port: the reference's JAX/TFP stack cannot be
           installed here, SURVEY 8c) on all host cores, on a bounded candidate sample.
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

SEED = 0
WORKLOADS = {
    # name: (N trials, D, total candidates (None = per GPU), candidates per GPU (None = total / world), scaling)
    'c2': dict(n=1000, d=20, m_per_gpu=100_000, m_total=None, scaling='weak'),
    'c5': dict(n=2000, d=50, m_per_gpu=None, m_total=1_000_000, scaling='strong'),
}
N_TRIALS, DIM, M_POOL = 1000, 20, 100_000   # the headline configuration (c2)


def make_problem(n=N_TRIALS, d=DIM):
  rng = np.random.default_rng(SEED)
  x = rng.uniform(size=(n, d))
  y = -np.sum((x - 0.3) ** 2, axis=1) + 0.05 * rng.normal(size=n)
  ls2 = 0.5 * (1 + np.arange(d) / d)
  return x, y, dict(sf2=1.0, ls2=ls2, sn2=1e-3)


def algorithmic_flops_per_candidate(n, d):
  # triangular contraction N^2 (N^2/2 FMA: L^-1 is lower triangular, what the reference's triangular_solve
  # does as well) + kernel row N*(3D+25) + mean 2N  (DESIGN.md section 4; SURVEY 8d counts a dense 2N^2)
  return n * n + n * (3 * d + 25) + 2 * n


def algorithmic_bytes_per_candidate(d):
  return 8 * d + 8


def fp64_peak_tflops():
  p = os.path.join(ROOT, 'profiles', 'fp64_peak_r01.json')
  if os.path.exists(p):
    try:
      j = json.load(open(p))
      return float(max(j['dfma_tflops'], j['dmma_m8n8k4_tflops'])), 'measured (tools/fp64_peak.cu, profiles/fp64_peak_r01.json)'
    except Exception:  # pylint: disable=broad-except
      pass
  return 37.0, 'nominal B200 FP64 (no measurement found)'


def int8_peak_tops():
  """Dense int8 tensor roof.  tcgen05 kind::i8 runs at the fp8 rate = 2 x bf16 (tools/umma_rate.cu: identical cycles per
  MMA for i8 and f8f6f4 at equal bytes); MEASURED_PEAKS.json carries the measured bf16 figure - the sustained one, the
  kernel is timed inside a long step."""
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    try:
      j = json.load(open(p))
      return 2.0 * float(j.get('bf16_tflops_sustained', j['bf16_tflops'])), '2 x measured sustained dense bf16 (MEASURED_PEAKS.json)'
    except Exception:  # pylint: disable=broad-except
      pass
  return 2.0 * 1590.0, '2 x the fallback dense bf16 figure of B200_PROFILING.md (1.59 PFLOP/s)'


def i8_ops_per_candidate(n):
  # 28 digit-pair products (7 x 7 balanced base-256 digits, s + t <= 8) of the triangular contraction: n(n+1)/2 MACs each
  return 28 * n * (n + 1)


def hbm_peak_gbs():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    try:
      return float(json.load(open(p))['hbm_gbs']), 'measured'
    except Exception:  # pylint: disable=broad-except
      pass
  return 6650.0, 'fallback'


def score_kernel_traffic(i8=False):
  """dram__bytes_read.sum + dram__bytes_write.sum of one k_score launch (ncu --set full), newest summary."""
  for name in (('score_i8_kernel_ncu_r02.json',) if i8 else ('score_kernel_ncu_r02.json', 'score_kernel_ncu_r01_latest.json')):
    tp = os.path.join(ROOT, 'profiles', name)
    if not os.path.exists(tp):
      continue
    try:
      j = json.load(open(tp))

      def _b(k):
        v, u = float(j[k]['value']), j[k]['unit'].lower()
        return v * {'gbyte': 1e9, 'mbyte': 1e6, 'kbyte': 1e3, 'byte': 1.0}[u]
      return _b('dram__bytes_read.sum') + _b('dram__bytes_write.sum'), name
    except Exception:  # pylint: disable=broad-except
      continue
  return None, None


class ClockSampler:
  """nvidia-smi clocks/throttle reasons during the timed region."""

  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index):
    self.gpu = gpu_index
    self.lines = []
    self.proc = None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '50'],
          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._read, daemon=True)
      self.t.start()
    except Exception:  # pylint: disable=broad-except
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def stop(self):
    if not self.proc:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:  # pylint: disable=broad-except
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    for ln in self.lines:
      f = [s.strip() for s in ln.split(',')]
      if len(f) < 9:
        continue
      try:
        sm.append(float(f[1])); mx.append(float(f[2]))
      except ValueError:
        continue
      for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], f[5:9]):
        if v.lower().startswith('active'):
          reasons.add(name)
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle on every host core
# --------------------------------------------------------------------------------------------------
def _host_cores():
  try:
    return max(1, len(os.sched_getaffinity(0)))
  except AttributeError:
    return os.cpu_count() or 1


_CPU_PRED = None


def _cpu_worker_init(n, d):
  """Worker process of the CPU arm: BLAS pinned to one thread, the oracle's predictive built once."""
  global _CPU_PRED
  for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
    os.environ[k] = '1'
  try:
    from threadpoolctl import threadpool_limits
    threadpool_limits(limits=1, user_api='blas')
  except Exception:  # pylint: disable=broad-except
    pass
  from oracle import gp_oracle as go
  x, y, th = make_problem(n, d)
  _CPU_PRED = go.precompute_predictive(go.GPParams(th['sf2'], th['ls2'], th['sn2']), x, y)


def _cpu_worker(chunk):
  from oracle import gp_oracle as go
  return float(np.sum(go.score_with_aux(_CPU_PRED, chunk)[0]))


class CpuArm:
  """The oracle (NumPy/SciPy) on EVERY host core: one worker PROCESS per core (spawned: no GIL, no allocator
  lock shared between workers, no CUDA state), BLAS pinned to one thread per worker.  A pass scores a bounded
  sample of the workload, `cores` chunks of `rows_per_worker` candidates; pool start-up and one warm-up pass
  happen in __enter__, outside every timed pass."""

  def __init__(self, n=N_TRIALS, d=DIM, rows_per_worker=512):
    self.n, self.d, self.rows = n, d, rows_per_worker
    self.cores = _host_cores()
    self.sample = self.cores * rows_per_worker
    xs = np.random.default_rng(1).uniform(size=(self.sample, d))
    self.chunks = [xs[i:i + rows_per_worker] for i in range(0, self.sample, rows_per_worker)]

  def __enter__(self):
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor
    self.ex = ProcessPoolExecutor(max_workers=self.cores, mp_context=mp.get_context('spawn'),
                                  initializer=_cpu_worker_init, initargs=(self.n, self.d))
    list(self.ex.map(_cpu_worker, self.chunks))   # every worker imports, builds its predictive, scores once
    return self

  def __exit__(self, *exc):
    self.ex.shutdown()

  def one_pass(self):
    """Seconds for one pass over the sample."""
    t0 = time.perf_counter()
    list(self.ex.map(_cpu_worker, self.chunks))
    return time.perf_counter() - t0


def cpu_oracle_rate(reps, n=N_TRIALS, d=DIM, rows_per_worker=512):
  """(candidates/s, seconds per pass, workers used, sample size) of the CPU arm, `reps` timed passes."""
  with CpuArm(n, d, rows_per_worker) as arm:
    dt = float(np.mean([arm.one_pass() for _ in range(reps)]))
    return arm.sample / dt, dt, min(arm.cores, len(arm.chunks)), arm.sample


def cpu_suggest_oracle(x, y, budget_s=60.0):
  """The designer's suggest() pipeline restated on the CPU with the oracle: 4 x 50 L-BFGS-B ARD (restarts
  one after the other like jaxopt_wrappers.py:139-152, BLAS on all cores), precompute_predictive, score an
  M=100k random pool + top-1 (rate from `cpu_oracle_rate`, all cores).  ARD is cut off after `budget_s`
  seconds and extrapolated over the remaining restarts (flagged)."""
  from oracle import gp_oracle as go
  from vizier_b200 import output_warpers   # host NumPy label warping, the same as the designer applies
  y = output_warpers.create_default_warper().warp(np.asarray(y, np.float64)[:, None])[:, 0]
  rng = np.random.default_rng(7)
  n, d = x.shape
  out = {}
  t0 = time.perf_counter()
  done, evals = 0, 0
  best, best_loss = None, np.inf

  def counted(theta, *a):
    nonlocal evals
    evals += 1
    return go.loss_and_grad(theta, *a)

  import scipy.optimize as sopt
  lo, hi = go.param_bounds(d, 0)
  for _ in range(4):
    t_init = go.log_uniform_init(rng, d, 0)
    res = sopt.minimize(counted, t_init, args=(x, y), jac=True, method='L-BFGS-B', bounds=list(zip(lo, hi)),
                        options={'maxiter': 50, 'gtol': 1e-8, 'maxls': 20})
    done += 1
    if res.fun < best_loss:
      best, best_loss = res.x, res.fun
    if time.perf_counter() - t0 > budget_s:
      break
  ard_s = time.perf_counter() - t0
  out['ard_restarts_run'] = done
  out['ard_evaluations'] = evals
  out['ard_extrapolated'] = done < 4
  out['ard_s'] = ard_s * 4 / done
  t0 = time.perf_counter()
  go.precompute_predictive(go.GPParams.from_vector(best, d, 0), x, y)
  out['fit_s'] = time.perf_counter() - t0
  rate, _, cores, sample = cpu_oracle_rate(2)
  out['score_100k_s'] = M_POOL / rate
  out['score_sample'] = sample
  out['cores'] = cores
  out['total_s'] = out['ard_s'] + out['fit_s'] + out['score_100k_s']
  return out


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  with CpuArm() as arm:
    for _ in range(args.warmup):
      arm.one_pass()
    t_all = float(np.sum([arm.one_pass() for _ in range(args.steps)]))
    cores, sample = min(arm.cores, len(arm.chunks)), arm.sample
  v = sample * args.steps / t_all
  line = {
      'impl': 'reference', 'metric': 'GP-UCB candidates scored/sec', 'value': v, 'unit': 'candidates/s',
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t_all / args.steps,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
      'config': {'workload': f'C2: GP posterior mu/var + UCB, N={N_TRIALS}, D={DIM}, M={M_POOL} (CPU arm: bounded sample of {sample} candidates per step)'},
      'cpu_baseline': {'value': v, 'unit': 'candidates/s', 'cores': cores, 'kind': 'port',
                       'sample': f'{sample} candidates/step = {cores} worker processes x 512 rows, NumPy/SciPy oracle (reference JAX/TFP build unavailable)'},
      'e2e': {'value': v, 'unit': 'candidates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# suggest() end to end (N = 1): the metric's second half
# --------------------------------------------------------------------------------------------------
def suggest_e2e_leg(device_index, reps=3):
  from vizier_b200 import optimizers as vb
  from vizier_b200 import profiler, vz
  from vizier_b200.designers import gp_bandit

  def problem():
    p = vz.ProblemStatement()
    for i in range(DIM):
      p.search_space.root.add_float_param(f'x{i}', 0.0, 1.0)
    p.metric_information.append(vz.MetricInformation(name='obj', goal=vz.ObjectiveMetricGoal.MAXIMIZE))
    return p

  def trials(xs, ys, first_id):
    out = []
    for i, (x, yv) in enumerate(zip(xs, ys)):
      t = vz.Trial(parameters={f'x{j}': float(x[j]) for j in range(DIM)}, id=first_id + i)
      t.complete(vz.Measurement({'obj': float(yv)}))
      out.append(t)
    return out

  x, y, _ = make_problem()
  rng = np.random.default_rng(99)
  res = {}
  pool_factory = vb.VectorizedOptimizerFactory(strategy_factory=vb.random_strategy_factory, max_evaluations=M_POOL,
                                               suggestion_batch_size=M_POOL)
  for name, kwargs in (('random_pool_100k', dict(acquisition_optimizer_factory=pool_factory)), ('eagle_default', {})):
    d = gp_bandit.VizierGPBandit(problem(), rng=1, device=device_index, **kwargs)
    d.update(vz.CompletedTrials(trials(x, y, 1)), vz.ActiveTrials())
    d.suggest(1)                                   # first call: workspaces, worker handles, graphs
    times, parts = [], []
    for r in range(reps):
      xn = rng.uniform(size=(1, DIM))
      yn = -np.sum((xn - 0.3) ** 2, axis=1) + 0.05 * rng.normal(size=1)
      d.update(vz.CompletedTrials(trials(xn, yn, N_TRIALS + 1 + r)), vz.ActiveTrials())   # one new trial -> refit
      with profiler.collect_events() as ev:
        t0 = time.perf_counter(); d.suggest(1); times.append(time.perf_counter() - t0)
      parts.append({k.split('.')[-1]: float(np.sum(v)) for k, v in ev.items()})
    k = int(np.argsort(times)[len(times) // 2])
    res[name] = {'gpu_s': float(times[k]), 'all_s': [float(t) for t in times],
                 'breakdown_s': {'convert': parts[k].get('_trials_to_data'), 'ard_and_fit': parts[k].get('_update_gp'),
                                 'optimize_acquisition': parts[k].get('_optimize_acquisition')}}
  cpu = cpu_suggest_oracle(x, y)
  out = {'config': f'VizierGPBandit.suggest(1), {N_TRIALS} completed {DIM}-D trials + 1 new trial, ARD 4 restarts x 50 L-BFGS-B iterations',
         'gpu_s': res['random_pool_100k']['gpu_s'], 'cpu_s': cpu['total_s'],
         'speedup': cpu['total_s'] / res['random_pool_100k']['gpu_s'],
         'breakdown': res['random_pool_100k']['breakdown_s'], 'gpu': res,
         'cpu': dict(cpu, kind='port', note='NumPy/SciPy oracle restatement of the same pipeline on the host cores; '
                     'the reference JAX/TFP build is not installable here')}
  return out


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, arrays):
  """Writes each array as out_dir/<name>.npy (float64), so that two builds can be compared output for output."""
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, f'{name}.npy'), np.asarray(a, dtype=np.float64))


def run_gpu(args):
  import torch
  from vizier_b200 import gp

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  dist = None
  if world > 1:
    import torch.distributed as dist  # pylint: disable=g-import-not-at-top
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  torch.cuda.set_device(local)
  wl = WORKLOADS[args.workload]
  n_trials, dim = wl['n'], wl['d']
  m_pool = wl['m_per_gpu'] if wl['m_per_gpu'] else wl['m_total'] // world
  dev = gp.DeviceGP(local)
  x, y, th = make_problem(n_trials, dim)
  params = gp.GPHyperParams(th['sf2'], th['ls2'], th['sn2'])
  dev.fit(x, y, params)  # every rank recomputes the (deterministic) factorisation: no broadcast needed
  from vizier_b200.multi_gpu import trust_radius, TopkExchange
  acq = gp.Acquisition(1.8, True, trust_radius(n_trials, dim, 0))

  # rotating candidate pools, together larger than the 126 MB L2, so no step re-reads its inputs from L2
  pool_bytes = m_pool * dim * 8
  n_pools = max(2, int(np.ceil(160e6 / pool_bytes)))
  pools = [dev.random_pool(m_pool, dim, seed=SEED + 17, index_base=(rank * n_pools + i) * m_pool)
           for i in range(n_pools)]
  n_slots = 8
  outs = [torch.empty(m_pool, dtype=torch.float64, device=dev.device) for _ in range(2)]
  stream = dev.stream
  exchange = TopkExchange(dist, dev, dim, 1, slots=n_slots)
  state = {'read': 0}

  def base(i):
    return (rank * n_pools + i % n_pools) * m_pool

  def step(i):
    # one suggest over this rank's shard, all on the handle's stream with no host synchronisation:
    # fused score -> device top-1 -> pack [score, global index, x] -> ONE fused kernel (push to all peers
    # over NVLink, flags, merge) -> async D2H of the winner.  The host reads winners n_slots-1 steps
    # behind, so a late host thread does not stall the device (or the other ranks) for up to 7 steps.
    exchange.step(i % n_slots, pools[i % n_pools], acq, index_base=base(i), score_out=outs[i % 2])
    if i >= n_slots - 1:
      state['winner'] = exchange.result((i - (n_slots - 1)) % n_slots)
      state['read'] += 1

  def drain(total):
    for j in range(max(0, total - (n_slots - 1)), total):
      state['winner'] = exchange.result(j % n_slots)

  for i in range(args.warmup):
    step(i)
  drain(args.warmup)
  dev.synchronize()
  step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
  if dist is not None:
    dist.barrier()
  torch.cuda.synchronize()
  sampler = ClockSampler(local)
  if rank == 0:
    if not args.no_cpu: sampler.start()
  l0 = dev.launch_count
  step_ev[0].record(stream)
  for i in range(args.steps):
    step(i)
    step_ev[i + 1].record(stream)
  drain(args.steps)
  torch.cuda.synchronize()
  if args.dump_outputs:
    # read now: the legs below overwrite the score buffers
    w_idx, w_val, w_x = state['winner']
    dumped = {'scores' if world == 1 else f'scores_rank{rank}': outs[(args.steps - 1) % 2].cpu().numpy()}
    if rank == 0:
      dumped.update(winner_index=w_idx.astype(np.float64), winner_score=w_val, winner_x=w_x)
    dump_outputs(args.dump_outputs, dumped)
  if dist is not None:
    dist.barrier()
  launches = dev.launch_count - l0
  total_ms = step_ev[0].elapsed_time(step_ev[-1])
  per_step = np.array([step_ev[i].elapsed_time(step_ev[i + 1]) for i in range(args.steps)])
  exchange_ok = exchange.peer.status() == 0 if exchange.peer is not None else True

  # latency of ONE synchronous suggest (enqueue -> winner on the host), median of 5
  lat = []
  for i in range(5):
    if dist is not None:
      dist.barrier()
    t0 = time.perf_counter()
    exchange.step(0, pools[i % n_pools], acq, index_base=base(i), score_out=outs[0])
    w_idx, w_val, _ = exchange.result(0)
    lat.append(1e3 * (time.perf_counter() - t0))
  suggest_latency_ms = float(np.median(lat))
  ranks_agree = True
  if dist is not None:   # every rank must have merged the same global winner
    mine = torch.tensor([float(w_idx[0]), float(w_val[0])], dtype=torch.float64, device=dev.device)
    allw = torch.empty((world, 2), dtype=torch.float64, device=dev.device)
    dist.all_gather_into_tensor(allw, mine)
    ranks_agree = bool((allw == allw[0]).all().item())

  # duration of the dominant kernel alone: CUDA events on the launching stream around each launch
  ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
  out_k = {'score': outs[0]}
  for i in range(args.steps):
    ev[i][0].record(stream)
    dev.score(pools[i % n_pools], acq, out=out_k)
    ev[i][1].record(stream)
  torch.cuda.synchronize()
  kern_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
  # which kernel that was: the tcgen05 integer-split kernel (default for pools of this size) or the FP64 DMMA kernel
  i8_before = dev.get_int('score_i8_launches')
  dev.score(pools[0], acq, out=out_k)
  used_i8 = dev.get_int('score_i8_launches') > i8_before
  dmma_ms = kern_ms
  if used_i8:   # the DMMA kernel on the same pools, for the record (round 1's dominant kernel)
    dev.set_int('score_i8', 0)
    for i in range(3):
      dev.score(pools[i % n_pools], acq, out=out_k)
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(args.steps, 10))]
    for i, (a_, b_) in enumerate(ev2):
      a_.record(stream)
      dev.score(pools[i % n_pools], acq, out=out_k)
      b_.record(stream)
    torch.cuda.synchronize()
    dmma_ms = float(np.mean([a_.elapsed_time(b_) for a_, b_ in ev2]))
    dev.set_int('score_i8', -1)
  # the trust-region variant k_score<true> (active when the radius is <= 0.5: few trials), same pool size
  tr_ms = None
  if args.workload == 'c2' and rank == 0:
    n_tr = 100
    dev_tr = gp.DeviceGP(local)
    dev_tr.fit(x[:n_tr], y[:n_tr], params)
    acq_tr = gp.Acquisition(1.8, True, trust_radius(n_tr, dim, 0))
    o_tr = {'score': outs[1]}
    for _ in range(3):
      dev_tr.score(pools[0], acq_tr, out=o_tr)
    dev_tr.synchronize()
    ts = []
    for i in range(10):
      a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a_.record(dev_tr.stream); dev_tr.score(pools[i % n_pools], acq_tr, out=o_tr); b_.record(dev_tr.stream)
      dev_tr.synchronize(); ts.append(a_.elapsed_time(b_))
    tr_ms = {'n_trials': n_tr, 'trust_radius': acq_tr.trust_radius, 'kernel': 'k_score<true>', 'ms': float(np.mean(ts)),
             'candidates_per_s': m_pool / (float(np.mean(ts)) * 1e-3)}
    dev_tr.close()

  # ---- e2e: one C-ABI call per step with HOST buffers, the collective included ----
  host_x = [torch.empty((m_pool, dim), dtype=torch.float64).pin_memory() for _ in range(2)]
  host_s = torch.empty(m_pool, dtype=torch.float64).pin_memory()
  for i in range(2):
    host_x[i].copy_(pools[i].cpu())
  for i in range(max(1, args.warmup)):
    dev.suggest_host(host_x[i % 2], acq, 1, base(i), exchange=exchange.peer, score_out=host_s)
  torch.cuda.synchronize()
  if dist is not None:
    dist.barrier()
  t0 = time.perf_counter()
  for i in range(args.steps):
    dev.suggest_host(host_x[i % 2], acq, 1, base(i), exchange=exchange.peer, score_out=host_s)
  torch.cuda.synchronize()
  e2e_s = time.perf_counter() - t0
  clocks = sampler.stop() if rank == 0 else None

  per_rank = None
  if dist is not None:
    t = torch.tensor([total_ms, kern_ms, e2e_s * 1e3, dmma_ms], dtype=torch.float64, device=dev.device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_ms, e2e_ms, dmma_ms = [float(v) for v in t.cpu()]
    e2e_s = e2e_ms / 1e3
    mine = torch.tensor([per_step.min(), float(np.median(per_step)), per_step.max(), float(np.argmax(per_step)),
                         1.0 if exchange_ok else 0.0], dtype=torch.float64, device=dev.device)
    allp = torch.empty((world, 5), dtype=torch.float64, device=dev.device)
    dist.all_gather_into_tensor(allp, mine)
    per_rank = allp.cpu().numpy()
    exchange_ok = bool(per_rank[:, 4].min() > 0)
  if rank != 0:
    if dist is not None:
      dist.destroy_process_group()
    return

  if per_rank is None:
    per_rank = np.array([[per_step.min(), np.median(per_step), per_step.max(), np.argmax(per_step), 1.0]])
  worst = int(np.argmax(per_rank[:, 2]))
  step_stats = {'min': float(per_rank[:, 0].min()), 'median': float(np.median(per_rank[:, 1])),
                'max': float(per_rank[:, 2].max()), 'max_rank': worst, 'max_step': int(per_rank[worst, 3]),
                'note': 'CUDA-event time of each step on each rank; min / median-of-medians / max over ranks'}
  cand_total = m_pool * world * args.steps
  value = cand_total / (total_ms * 1e-3)
  flops = algorithmic_flops_per_candidate(n_trials, dim) * m_pool
  peak, peak_src = fp64_peak_tflops()
  achieved = flops / (dmma_ms * 1e-3) * 1e-12
  hbm_peak, hbm_src = hbm_peak_gbs()
  hbm_ach = algorithmic_bytes_per_candidate(dim) * m_pool / (kern_ms * 1e-3) * 1e-9
  traffic, traffic_src = score_kernel_traffic(used_i8) if args.workload == 'c2' else (None, None)
  dmma_roof = {'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
               'kernel': 'k_score', 'kernel_ms': dmma_ms,
               'note': 'the FP64 DMMA kernel (mma.sync m8n8k4 f64) on the same pools; peak ' + peak_src}
  if used_i8:
    i8_peak, i8_src = int8_peak_tops()
    i8_ach = i8_ops_per_candidate(n_trials) * m_pool / (kern_ms * 1e-3) * 1e-12
    roofline = {'bound': 'tensor', 'achieved': i8_ach, 'peak': i8_peak, 'unit': 'TOP/s', 'frac': i8_ach / i8_peak,
                'traffic': traffic, 'traffic_source': traffic_src, 'kernel': 'k_score_i8', 'kernel_ms': kern_ms,
                'note': 'frac is against the INT8 tensor roof of the kernel that now runs; measured against round 1\'s FP64 DMMA roof '
                        '(frac 0.755 then) the same work is fp64_equivalent.of_fp64_dmma_peak.  '
                        'tcgen05.mma kind::i8 (s8 x s8 -> s32 in TMEM): W = K* Linv^T as 28 exact products of balanced base-256 '
                        'digit planes, recombined in fp64; peak = ' + i8_src + '.  M = 128, N = 64 MMAs (7 accumulator groups x 64 '
                        'columns fill TMEM) read 6 KB of shared memory per 32-cycle MMA: the operand bandwidth bounds them at 48 '
                        'cycles = 0.67 of the tensor peak (tools/umma_rate.cu)',
                'int8_ops_per_candidate': i8_ops_per_candidate(n_trials),
                'fp64_equivalent': {'tflops': flops / (kern_ms * 1e-3) * 1e-12, 'of_fp64_dmma_peak': flops / (kern_ms * 1e-3) * 1e-12 / peak,
                                    'flops_per_candidate': algorithmic_flops_per_candidate(n_trials, dim)},
                'fp64_dmma_kernel': dmma_roof,
                'hbm': {'achieved': hbm_ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': hbm_ach / hbm_peak, 'peak_source': hbm_src}}
  else:
    roofline = dict(dmma_roof, traffic=traffic, traffic_source=traffic_src,
                    note='fp64: tcgen05 has no f64 kind, the binding roof is the FP64 DMMA pipe; peak ' + peak_src,
                    flops_per_candidate=algorithmic_flops_per_candidate(n_trials, dim),
                    hbm={'achieved': hbm_ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': hbm_ach / hbm_peak, 'peak_source': hbm_src})
  cname = args.workload.upper()
  line = {
      'metric': 'GP-UCB candidates scored/sec', 'value': value, 'unit': 'candidates/s', 'n_gpus': world,
      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms / args.steps,
      'higher_is_better': True, 'scaling': wl['scaling'], 'vs_baseline': None, 'dtype': 'f64 (W = K* Linv^T as exact s8 digit products on tcgen05)' if used_i8 else 'f64', 'data': 'synthetic',
      'config': {'workload': f'{cname}: GP posterior mu/var + UCB + trust region + top-1, N={n_trials}, D={dim}, M={m_pool} per GPU'
                             + (f' ({wl["m_total"]} in total)' if wl['m_total'] else ''),
                 'l2': f'{n_pools} rotating candidate pools ({n_pools * pool_bytes / 1e6:.0f} MB > 126 MB L2)',
                 'parallelism': (f'candidate-pool shards x{world}; global arg-max by ONE fused kernel per step (NVLink peer stores + '
                                 f'release/acquire flags + merge), transport={exchange.transport}') if world > 1 else 'single GPU',
                 'suggest_latency_ms': suggest_latency_ms, 'ranks_agree': ranks_agree, 'exchange_ok': exchange_ok,
                 'per_step_ms': step_stats,
                 'pipelining': f'steps are enqueued without host sync; the host reads winners {n_slots - 1} steps behind',
                 'k_score_trust_region_variant': tr_ms},
      'roofline': roofline,
      'e2e': {'value': m_pool * world * args.steps / e2e_s, 'unit': 'candidates/s',
              'h2d_bytes_per_step': m_pool * dim * 8 * world, 'd2h_bytes_per_step': (m_pool * 8 + (dim + 2) * 8) * world,
              'ms_per_step': 1e3 * e2e_s / args.steps,
              'call': 'vzgp_suggest_host: H2D candidates, score, top-1, exchange+merge, D2H scores + winner, host-synchronous'},
      'gpu_launches': int(launches),
      'clocks': clocks,
  }
  if world == 1 and args.workload == 'c2' and not args.no_cpu:
    cpu_v, cpu_dt, cores, sample = cpu_oracle_rate(3)
    line['cpu_baseline'] = {'value': cpu_v, 'unit': 'candidates/s', 'cores': cores, 'kind': 'port',
                            'sample': f'{sample} candidates x 3 passes ({cpu_dt:.2f} s each): {cores} worker processes x 512 rows, '
                                      'NumPy/SciPy oracle, one process per core'}
    if not args.no_suggest:
      try:
        line['suggest_e2e'] = suggest_e2e_leg(local)
      except Exception as e:  # pylint: disable=broad-except
        line['suggest_e2e'] = {'error': repr(e)}
  print(json.dumps(line), flush=True)
  if dist is not None:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=50)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
  ap.add_argument('--no-suggest', action='store_true', help='skip the suggest() end-to-end leg (N=1)')
  ap.add_argument('--no-cpu', action='store_true',
                  help='skip the cpu_baseline leg and everything that spawns processes (runs under ncu)')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='after the timed steps, write what the last one returned to DIR/<name>.npy (float64): '
                       'scores (this rank\'s candidate scores; scores_rank<r> when there are several ranks), '
                       'winner_index, winner_score and winner_x (the merged global arg-max)')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'b200':
    ap.error('--dump-outputs writes the outputs of the GPU path (--impl b200)')
  args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_gpu(args)


if __name__ == '__main__':
  main()
