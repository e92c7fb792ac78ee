#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched RAMP cluster simulator hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # product arm (CUDA kernels through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the unmodified Python reference (oracle/_ref), one
                                                              # process per core; the C port of its algorithm beside it

One bench "step" = one batched env-step: every one of the B episodes takes one agent decision, i.e. one
``RampClusterEnvironment.step(action)`` plus the ``step(Action())`` calls until the next job is queued
(RJPE:300-420).  Episodes are scripted rollouts of L decisions each (ddls_b200/workload.py); every L steps
all episodes are reset (which clears the per-episode memo tables like RCE:269-275), so the timed region
contains resets, memo misses (lookaheads executed) and memo hits in the proportion a real rollout has.

Prints ONE JSON line (rank 0).  See README / DESIGN.md for the field definitions.
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
# rank 0 must print ONE JSON line on stdout.  NCCL's log (whatever NCCL_DEBUG level the caller asked for) goes to stderr, and so
# does anything a library printf()s to file descriptor 1 (NCCL prints its version banner there when NCCL_DEBUG is unset): the
# real stdout is kept aside and only emit() writes to it.
if not os.environ.get('NCCL_DEBUG_FILE'):
    os.environ['NCCL_DEBUG_FILE'] = '/dev/stderr'
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)
sys.stdout = os.fdopen(os.dup(2), 'w', buffering=1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + '\n').encode())

METRIC = 'env_steps_per_sec'
UNIT = 'env-steps/s'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=256)
    ap.add_argument('--warmup', type=int, default=16)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='cfg3-resnet50-64w')
    ap.add_argument('--episodes', type=int, default=0, help='episodes per GPU (0 = the config\'s batch size)')
    ap.add_argument('--segment', type=int, default=8, help='L: agent decisions per scripted episode')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--cpu-sample', type=int, default=0, help='episodes in the CPU baseline sample (0 = auto)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--memo-mode', type=int, default=0)
    ap.add_argument('--run-times', default='reference', choices=['reference', 'one_to_one'],
                    help="dep run times of the scripted jobs: 'reference' = the reference pipeline's lowered jobs on an empty cluster "
                         "(collectives; T=1,334 for the degree-16 bench job), 'one_to_one' = round 1's lighter stand-in (T=1,169)")
    ap.add_argument('--ref-budget', type=float, default=90.0, help='--impl reference: seconds of timed env-steps per process')
    ap.add_argument('--ref-procs', type=int, default=0, help='--impl reference: processes (0 = min(usable cores, 32))')
    ap.add_argument('--ref-kind', default='auto', choices=['auto', 'reference', 'port'])
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: --episodes (or the config batch) per GPU; strong: the config batch divided over the GPUs')
    ap.add_argument('--gather-every', type=int, default=0,
                    help='all-gather the episode metrics every this many steps (0 = once per scripted segment, i.e. per batch of rollouts)')
    ap.add_argument('--no-batched-env', action='store_true', help='skip the BatchedRampJobPartitioningEnvironment secondary figure')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned to its caller (rank 0) as DIR/step_stats.npy [B, STEP_STATS_LEN] '
                         'and DIR/cluster_steps.npy [B], float64; the inputs are a function of the arguments, so two builds can '
                         'be compared output for output')
    return ap.parse_args()


def dump_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f'{name}.npy'), a)


def usable_cores():
    """Host threads this process may really use: the scheduler affinity mask capped by the cgroup CPU quota (a leased box can
    report 128 CPUs in os.cpu_count() and still be limited to a fraction of them)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:                       # cgroup v2
            q, per = f.read().split()
            if q != 'max':
                quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())  # cgroup v1
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return {'affinity': n, 'cgroup_quota': quota, 'os_cpu_count': os.cpu_count(), 'used': eff}


def workload_config(args, cfg, templates, world, B):
    """The `config` object of the JSON line: the same keys for the product arm and the reference arm."""
    return {'workload': args.config, 'episodes_per_gpu': B, 'segment': args.segment,
            'cluster': 'x'.join(map(str, cfg['shape'])) + ' RAMP', 'degrees': list(cfg['degrees']),
            'templates': [[t.n_ops, t.n_deps] for t in templates], 'run_times': args.run_times, 'memo_mode': args.memo_mode,
            'agent': 'scripted: partition degree drawn from `degrees` + first-fit blocks -- the same decision rule in both arms; the same '
                     'rollouts driven by the GNN policy on the device are reported in batched_env.device_gnn_policy',
            # identical text in both arms so that the two `config` objects compare equal
            'l2': 'product arm: inputs larger than L2 are not needed -- the lookahead kernel keeps its working set (template blob + per-lane '
                  'lists) in shared memory and streams its tick traces to HBM (trace_mb_per_step in the line); no explicit flush.  '
                  'reference arm: CPU, not applicable',
            'parallelism': (f'product arm: episodes sharded x{world}, one process per GPU, one NCCL all-gather of episode metrics per batch of '
                            f'rollouts on a side stream (none at 1 GPU); reference arm: one single-threaded process per usable host core on rank 0')}


# ---------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): NVML when importable,
    else the nvidia-smi query line."""

    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0, period=0.2):
        super().__init__(daemon=True)
        self.gpu_index, self.period = gpu_index, period
        self.samples, self._stop_evt = [], threading.Event()

    def _nvml(self):
        """NVML handle for fast sampling (a 100 ms timed region gets ~1 nvidia-smi sample but tens of NVML ones)."""
        try:
            import pynvml
            pynvml.nvmlInit()
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
        except Exception:
            return None, None

    def run(self):
        nv, h = self._nvml()
        while not self._stop_evt.is_set():
            try:
                if nv is not None:
                    sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                    mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    act = lambda bit: 'Active' if (r & bit) else 'Not Active'
                    # bits: SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
                    self.samples.append([str(sm), str(mx), '', act(0x8), act(0x40), act(0x20), act(0x4)])
                    self._stop_evt.wait(0.01)
                    continue
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i',
                                      str(self.gpu_index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm, mx, reasons = [], 0.0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                continue
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def ncu_profile_summary():
    """STATIC figures from the committed ncu capture of this bench command (profiles/r2_ncu_thread_summary.json, written by
    scripts/ncu_summary.py): DRAM bytes per lookahead launch and warp instructions per lookahead.  Not measured in this run --
    counters need ncu, and a number taken under a profiler is never a bench value -- so they carry their source."""
    p = os.path.join(ROOT, 'profiles', 'r2_ncu_thread_summary.json')
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {'dram_bytes_per_launch': d.get('dram_bytes_per_launch'), 'warp_inst_per_lookahead': d.get('warp_inst_per_lookahead'),
                    'source': 'static, from profiles/r2_ncu_thread_summary.json'}
        except Exception:
            pass
    return {'source': 'no committed ncu summary'}


# ---------------------------------------------------------------------------------------------------------
def oracle_jcts(templates):
    from oracle import oracle
    oracle.build()
    return [oracle.run_lookahead(t, trace_cap=0)['jct'] for t in templates]


def run_reference_arm(args, rank, world):
    """The CPU arm.  kind "reference": the UNMODIFIED Python reference (staged at oracle/_ref by oracle/stage_ref.py, or
    the build container's checkout) -- RampJobPartitioningEnvironment with its own heuristic agents on the same
    topology / job graphs / degree rule, one process per core (the reference is single-threaded; RLlib runs one env per
    worker process), each taking --steps env-steps or as many as fit --ref-budget seconds (oracle/ref_runner.py).
    kind "port": oracle/ramp_oracle.c (the C restatement of the reference's algorithm) on all usable host threads, when the
    reference is not available.  The port's figure is always reported too (`port`), on the same scripted workload as the GPU arm."""
    if rank != 0:
        return
    from ddls_b200 import workload
    cores = usable_cores()
    cfg = workload.CONFIGS[args.config]
    B = args.episodes or cfg['n_episodes']
    L = args.segment
    templates = workload.build_templates(args.config, run_times=args.run_times)[3]
    config = workload_config(args, cfg, templates, world, B)
    port = port_throughput(args, cores['used'], budget_s=8.0)
    from oracle import ref_shim
    have_ref = ref_shim.reference_available()          # staged copy (oracle/_ref) or the build container's checkout
    kind = args.ref_kind if args.ref_kind != 'auto' else ('reference' if have_ref else 'port')
    if kind == 'reference' and not have_ref:
        kind = 'port'
    base = {'metric': METRIC, 'unit': UNIT, 'n_gpus': args.gpus, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic', 'impl': 'reference', 'config': config, 'host_cores': cores, 'port': port}
    if kind == 'port':
        value = port['value']
        line = dict(base, value=value, steps=args.steps, warmup=args.warmup, ms_per_step=B / value * 1e3,
                    cpu_baseline={'value': value, 'unit': UNIT, 'cores': cores['used'], 'kind': 'port', 'sample': port['sample'],
                                  'per_core': value / cores['used']},
                    e2e={'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0})
        emit(line)
        return
    P = args.ref_procs or max(1, min(cores['used'], 32))
    warm = 1 if args.warmup > 0 else 0
    t0 = time.perf_counter()
    procs = []
    for k in range(P):
        cmd = [sys.executable, os.path.join(ROOT, 'oracle', 'ref_runner.py'), '--config', args.config, '--steps', str(args.steps),
               '--warmup', str(warm), '--budget', str(args.ref_budget), '--seed', str(args.seed + k)]
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                      env=dict(os.environ, OMP_NUM_THREADS='1', MKL_NUM_THREADS='1', OPENBLAS_NUM_THREADS='1')))
    results, errors = [], []
    for pr in procs:
        out, err = pr.communicate()
        try:
            results.append(json.loads(out.strip().splitlines()[-1]))
        except Exception:
            errors.append((err or out)[-300:])
    wall = time.perf_counter() - t0
    if not results:
        raise RuntimeError('every reference process failed: ' + ' | '.join(errors[:3]))
    rates = [r['steps'] / r['elapsed_s'] for r in results]
    value = float(sum(rates))                                  # P independent single-threaded environments running side by side
    steps_min, steps_max = min(r['steps'] for r in results), max(r['steps'] for r in results)
    mean_s = float(np.mean([r['elapsed_s'] / r['steps'] for r in results]))
    line = dict(base, value=value, steps=steps_max, warmup=warm, ms_per_step=mean_s * 1e3,
                cpu_baseline={'value': value, 'unit': UNIT, 'cores': len(results), 'kind': 'reference', 'per_core': value / len(results),
                              'sample': f'{len(results)} processes x {steps_min}-{steps_max} env-steps of {args.config} each '
                                        f'({mean_s:.1f} s per env-step per process, budget {args.ref_budget:.0f} s, {wall:.0f} s wall incl. '
                                        f'imports and one warm-up step); unmodified reference from {results[0]["reference_root"]}',
                              'failed_processes': len(errors)},
                e2e={'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0})
    emit(line)


def port_throughput(args, n_threads, budget_s=10.0):
    """oracle/ramp_oracle.c on n_threads host threads over a bounded sample of the scripted workload: env-steps/s."""
    from oracle import oracle
    from ddls_b200 import workload
    oracle.build()
    L = args.segment
    S0 = max(n_threads, 16)
    wl = workload.generate(args.config, oracle_jcts, n_episodes=S0, n_steps=L, seed=args.seed, run_times=args.run_times)
    t0 = time.perf_counter()
    _oracle_segment(oracle, wl, n_threads)
    probe = time.perf_counter() - t0
    cap = args.episodes or workload.CONFIGS[args.config]['n_episodes']
    S = int(max(S0, min(max(cap, S0), S0 * (budget_s / 2) / max(probe, 1e-6))))
    S = max(n_threads, (S // n_threads) * n_threads)
    if S != S0:
        wl = workload.generate(args.config, oracle_jcts, n_episodes=S, n_steps=L, seed=args.seed, run_times=args.run_times)
        _oracle_segment(oracle, wl, n_threads)      # warm-up (page in, thread start)
    t0 = time.perf_counter()
    reps = 0
    while reps < 1 or (time.perf_counter() - t0) < budget_s / 2:
        _oracle_segment(oracle, wl, n_threads)
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    value = S * L / dt
    return {'value': value, 'unit': UNIT, 'cores': n_threads, 'kind': 'port', 'per_core': value / n_threads,
            'sample': f'{S} episodes x {L} env-steps of {args.config}, {reps} repetitions, {dt:.2f} s wall each on {n_threads} threads '
                      f'(oracle/ramp_oracle.c)'}


def _oracle_segment(oracle, wl, n_threads):
    """Runs every episode of the workload for its L decisions (+ empty steps) through the oracle env, threaded."""
    import ctypes as C
    L, B = wl.n_steps, wl.n_episodes
    lib = oracle.lib()
    ctemps = (oracle.CLoweredJob * len(wl.templates))(*[oracle.to_c(t) for t in wl.templates])
    keep = [oracle.to_c(t) for t in wl.templates]   # keep numpy arrays alive
    # script: per episode the oracle env needs explicit Action() steps between decisions; orc_run_scripted_batch
    # takes a flat script, so expand each decision into (decision, then up to `pad` empty steps) conservatively:
    # instead use the dedicated fused driver below
    tid = np.ascontiguousarray(wl.actions['template_id'].T, dtype=np.int32)          # [B, L]
    mount = np.zeros((B, L), dtype=oracle.MOUNT_DTYPE)
    for f in ('max_acceptable_jct', 'part_op_mem', 'part_dep_size', 'flow_size', 'n_mounted_workers', 'n_mounted_channels'):
        mount[f] = wl.actions[f].T
    arr = np.ascontiguousarray(wl.arrivals, dtype=oracle.ARRIVAL_DTYPE)
    n_models = max(wl.template_model) + 1
    rc = lib.orc_run_scripted_rjpe_batch(ctemps, len(wl.templates), B, L, tid.ctypes.data, mount.ctypes.data,
                                         arr.ctypes.data, L, float('inf'), wl.shape.n_workers, n_models, 1025,
                                         None, None, n_threads)
    assert rc == 0, rc
    del keep


# ---------------------------------------------------------------------------------------------------------
def run_b200_arm(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from ddls_b200 import engine, workload

    if not torch.cuda.is_available():
        raise RuntimeError('bench.py --impl b200 needs a CUDA device; there is no CPU fallback')
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    cfg = workload.CONFIGS[args.config]
    B = args.episodes or cfg['n_episodes']
    if args.scaling == 'strong':
        B = max(1, B // world)                 # total work fixed: the config's batch divided over the GPUs
    L = args.segment

    # ---- build templates, get their JCTs from the CUDA path, script the episodes ----
    eng = engine.RampEngine(n_episodes=B, n_cluster_workers=int(np.prod(cfg['shape'])), max_jobs=L, device=local_rank,
                            memo_mode=args.memo_mode, trace_cap=4096)
    tmap = {}

    def engine_jcts(templates):
        for i, t in enumerate(templates):
            tmap[i] = eng.register_template(t)
        res, _ = eng.run_lookaheads([tmap[i] for i in range(len(templates))])
        assert (res['status'] == 0).all()
        return res['jct']

    wl = workload.generate(args.config, engine_jcts, n_episodes=B, n_steps=L, seed=args.seed + 1000 * rank, run_times=args.run_times)
    actions_host = []
    for p in range(L):
        a = wl.actions[p].copy()
        placed = a['template_id'] >= 0
        a['template_id'][placed] = np.array([tmap[int(t)] for t in a['template_id'][placed]], dtype=np.int32)
        actions_host.append(a)
    # pinned host copies (e2e path) and device-resident copies (value path)
    pinned, on_dev = [], []
    for a in actions_host:
        t = torch.from_numpy(a.view(np.uint8).reshape(B, -1).copy()).pin_memory()
        pinned.append(t)
        on_dev.append(t.cuda())
    arrivals = wl.arrivals
    stats_dev = torch.empty((B, engine.STEP_STATS_LEN), dtype=torch.float64, device='cuda')
    ncs_dev = torch.empty(B, dtype=torch.int32, device='cuda')
    stats_pinned = torch.empty((B, engine.STEP_STATS_LEN), dtype=torch.float64).pin_memory()
    # episode metrics: exported on the engine stream into one of two buffers, all-gathered over NCCL on a SIDE stream so that the
    # collective of step s overlaps the lookaheads of step s + 1 (episodes shard with no other exchange, SURVEY.md 8e)
    ep_dev = [torch.empty((B, engine.EP_LEN), dtype=torch.float64, device='cuda') for _ in range(2)]
    gathered = [torch.empty((world * B, engine.EP_LEN), dtype=torch.float64, device='cuda') for _ in range(2)] if world > 1 else None
    ext = torch.cuda.ExternalStream(eng.stream, device=torch.device('cuda', local_rank))
    side = torch.cuda.Stream(device=torch.device('cuda', local_rank)) if world > 1 else None
    gather_events = [None, None]
    n_gathers = [0]
    torch.cuda.synchronize()

    def barrier():
        if side is not None:
            side.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_metrics():
        k = n_gathers[0] & 1
        n_gathers[0] += 1
        if world > 1 and gather_events[k] is not None:
            ext.wait_event(gather_events[k])          # the collective that last read this buffer has finished
        eng.export_episode_state_to(ep_dev[k].data_ptr())
        if world > 1:
            ev = torch.cuda.Event()
            ev.record(ext)
            with torch.cuda.stream(side):
                side.wait_event(ev)
                dist.all_gather_into_tensor(gathered[k], ep_dev[k])
                done_ev = torch.cuda.Event()
                done_ev.record(side)
            gather_events[k] = done_ev

    gather_every = args.gather_every or L       # one NCCL all-gather of episode metrics per batch of rollouts (north_star)
    memo_acc = {'lookups': 0, 'hits': 0, 'lookaheads': 0}
    memo_base = {'lookups': 0, 'hits': 0, 'lookaheads': 0}     # part of the current segment that belongs to the warm-up

    def fold_memo():
        m = eng.memo_stats()           # since the last reset
        for k in memo_acc:
            memo_acc[k] += m[k] - memo_base[k]
            memo_base[k] = 0

    def device_step(s):
        p = s % L
        if p == 0:
            if s > 0:
                fold_memo()
            eng.reset(arrivals)
        eng.step_device(on_dev[p].data_ptr(), True, stats_dev.data_ptr(), ncs_dev.data_ptr())
        if (s + 1) % gather_every == 0:
            gather_metrics()

    def host_step(s):
        p = s % L
        if p == 0:
            eng.reset(arrivals)
        # HOST buffers in, HOST stats out: H2D + D2H inside the call (ramp_step_host)
        rc = eng._L.ramp_step_host(eng._h, pinned[p].data_ptr(), 1, stats_pinned.data_ptr(), None)
        if rc != 0:
            engine._check(rc)
        if (s + 1) % gather_every == 0:
            gather_metrics()
        return float(stats_pinned[0, engine.SS['step_end_time']])

    W, K = args.warmup, args.steps
    # ---- value: inputs resident in HBM ----
    for s in range(W):
        device_step(s)
    barrier()
    eng.lookahead_kernel_time(reset=True)
    m0 = eng.memo_stats()
    for k in memo_acc:
        memo_acc[k] = 0
        memo_base[k] = m0[k]           # the current segment's counts so far are warm-up
    launches0 = eng.launch_count
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(ext)
    for s in range(W, W + K):
        device_step(s)
    e1.record(ext)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    dev_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    # the buffers are written again by the legs below: keep the last timed step's outputs now
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'step_stats': stats_dev.cpu().numpy().astype(np.float64),
                                         'cluster_steps': ncs_dev.cpu().numpy().astype(np.float64)})
    launches = eng.launch_count - launches0
    kt = eng.lookahead_kernel_time(reset=True)
    fold_memo()
    memo = dict(memo_acc)
    eng.check_status()
    # the episode resets inside the loop synchronise the stream, so wall time ~ device time; use the larger
    elapsed_ms = max(dev_ms, 0.0)
    el = torch.tensor([elapsed_ms, t_wall * 1e3], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    elapsed_ms, wall_ms = float(el[0]), float(el[1])
    value = world * B * K / (elapsed_ms / 1e3)

    # ---- e2e: through the host-buffer C-ABI call ----
    for s in range(W):
        host_step(s)
    barrier()
    t0 = time.perf_counter()
    for s in range(W, W + K):
        host_step(s)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / float(e2e_t[0])
    eng.check_status()

    # ---- raw RampClusterEnvironment.step calls per env-step (SURVEY 8d): the scripted segments are deterministic, so one
    #      untimed replay of a segment counts them exactly (an env-step = 1 cluster.step(action) + k cluster.step(Action())) ----
    eng.reset(arrivals)
    n_cluster_steps = 0
    for p in range(L):
        eng.step_device(on_dev[p].data_ptr(), True, stats_dev.data_ptr(), ncs_dev.data_ptr())
        eng.sync()
        n_cluster_steps += int(ncs_dev.sum().item())
    cluster_steps_per_env_step = n_cluster_steps / float(B * L)

    # ---- secondary: RAMP_MEMO_SHARED (reference semantics + batch-wide result cache), device-resident inputs ----
    shared = None
    try:
        eng2 = engine.RampEngine(n_episodes=B, n_cluster_workers=int(np.prod(cfg['shape'])), max_jobs=L, device=local_rank,
                                 memo_mode=engine.MEMO_SHARED, trace_cap=4096)
        t2 = {i: eng2.register_template(t) for i, t in enumerate(wl.templates)}
        assert all(t2[i] == tmap[i] for i in t2)
        ext2 = torch.cuda.ExternalStream(eng2.stream, device=torch.device('cuda', local_rank))
        for s in range(W + K):
            if s == W:
                torch.cuda.synchronize()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record(ext2)
            if s % L == 0:
                eng2.reset(arrivals)
            eng2.step_device(on_dev[s % L].data_ptr(), True, stats_dev.data_ptr(), ncs_dev.data_ptr())
        f1.record(ext2)
        torch.cuda.synchronize()
        sh_ms = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(sh_ms, op=dist.ReduceOp.MAX)
        m2 = eng2.memo_stats_ex()
        shared = {'value': world * B * K / (float(sh_ms[0]) / 1e3), 'unit': UNIT, 'ms_per_step': float(sh_ms[0]) / K,
                  'memo_last_segment': m2,
                  'note': 'memo_mode=RAMP_MEMO_SHARED: per-episode reference semantics on top of a batch-wide result cache keyed by '
                          'the lowered job (identical results, tests/test_gpu_parity.py); NOT the headline: the CPU arm does not share'}
        eng2.close()
    except Exception as ex:          # secondary measurement only
        shared = {'error': str(ex)[:200]}

    # ---- secondary: the batched gym-like surface (ddls_b200/batched.py): RJPE.step for every episode through host arrays, with
    #      placement (native first-fit, cached by cluster occupancy), lowering (native expansion, cached by block) and the action
    #      mask / graph features computed on the host inside the timed region; policy stand-in: random valid degree ----
    batched = None
    if not args.no_batched_env:
        batched = {}
        from ddls_b200 import batched as batched_mod
        for label, cls in (('device', batched_mod.DeviceRampJobPartitioningEnvironment), ('host', batched_mod.BatchedRampJobPartitioningEnvironment)):
            try:
                graphs_b = [workload.make_graph(kind, **kw) for kind, kw in cfg['graphs']]
                benv = cls(tuple(cfg['shape']), graphs_b, n_episodes=B, jobs_per_episode=L, device=local_rank, seed=args.seed + 7 * rank,
                           run_times=args.run_times, interarrival=('exponential', 1000.0) if cfg.get('exponential') else ('fixed', 1000.0),
                           **({'prewarm': True} if label == 'device' else {}))
                degs = np.array([d for d in cfg['degrees'] if d <= benv.W])
                prng = np.random.default_rng(args.seed + 99 + rank)

                # the stand-in agent: a random valid degree per episode.  Its random numbers are drawn before the timed region (they
                # are the agent's, not the environment's); per step it only masks them and takes the row-wise maximum
                noise = np.ascontiguousarray((prng.random((min(K + max(W, L), 512), len(degs), benv.B), dtype=np.float32) + np.float32(1e-3)))
                step_no = [0]

                def policy(obs):
                    am, nz = obs['action_mask'], noise[step_no[0] % len(noise)]
                    step_no[0] += 1
                    best = np.where(am[:, degs[0]] != 0, nz[0], np.float32(0))
                    act = np.where(best > 0, degs[0], 0)
                    for j in range(1, len(degs)):
                        v = np.where(am[:, degs[j]] != 0, nz[j], np.float32(0))
                        act = np.where(v > best, degs[j], act)
                        np.maximum(best, v, out=best)
                    return act
                obs_b = benv.reset()
                for s_ in range(max(W, L)):               # at least one whole segment: every block geometry has been lowered once
                    if s_ % L == 0 and s_ > 0:
                        obs_b = benv.reset()
                    obs_b, _, _, _ = benv.step(policy(obs_b))
                calls0 = dict(benv.stats)
                barrier()
                tb = time.perf_counter()
                n_env_steps_b = 0
                for s_ in range(K):
                    if s_ % L == 0:
                        obs_b = benv.reset()
                    live_before = int((~obs_b['done']).sum())
                    obs_b, _, _, _ = benv.step(policy(obs_b))
                    n_env_steps_b += live_before
                barrier()
                tb = time.perf_counter() - tb
                tb_t = torch.tensor([tb], dtype=torch.float64, device='cuda')
                nb_t = torch.tensor([float(n_env_steps_b)], dtype=torch.float64, device='cuda')
                if world > 1:
                    dist.all_reduce(tb_t, op=dist.ReduceOp.MAX)
                    dist.all_reduce(nb_t, op=dist.ReduceOp.SUM)
                batched[label] = {'value': float(nb_t[0]) / float(tb_t[0]), 'unit': UNIT, 'ms_per_step': float(tb_t[0]) / K * 1e3,
                                  'native_placer_calls_in_timed_region': benv.stats['placer_calls'] - calls0['placer_calls'],
                                  'native_expansions_in_timed_region': benv.stats['expansions'] - calls0['expansions']}
                benv.close()
            except Exception as ex:
                batched[label] = {'error': repr(ex)[:300]}
        # ---- the same rollouts with the reference's GNN policy deciding on the device (ddls_b200/policy.py): sampled actions written
        #      straight into the environment's action buffer, no observation / reward / action crosses PCIe inside a segment ----
        try:
            from ddls_b200 import policy as policy_mod
            graphs_b = [workload.make_graph(kind, **kw) for kind, kw in cfg['graphs']]
            benv = batched_mod.DeviceRampJobPartitioningEnvironment(
                tuple(cfg['shape']), graphs_b, n_episodes=B, jobs_per_episode=L, device=local_rank, seed=args.seed + 7 * rank,
                run_times=args.run_times, interarrival=('exponential', 1000.0) if cfg.get('exponential') else ('fixed', 1000.0), prewarm=True)
            pol = policy_mod.DeviceGNNPolicy(graphs_b, benv.max_partitions_per_op + 1, device=local_rank, seed=args.seed)
            pol.embed()
            n_seg_w, n_seg = (max(W, L) + L - 1) // L, (K + L - 1) // L
            for g_ in range(n_seg_w):
                pol.collect(benv, L, sample=True, seed=args.seed + 100 * g_)
            barrier()
            tb = time.perf_counter()
            n_env_steps_b = 0
            for g_ in range(n_seg):
                # one segment = reset + L decisions of the policy per episode on the device, every decision recorded on the device
                # (observation, action, log-probability, value, reward, done) and read back ONCE: what a trainer consumes
                traj = pol.collect(benv, L, sample=True, seed=args.seed + 1000 + 100 * g_)
                n_env_steps_b += int(traj['live'].sum())
            barrier()
            tb = time.perf_counter() - tb
            K_pol = n_seg * L
            tb_t = torch.tensor([tb], dtype=torch.float64, device='cuda')
            nb_t = torch.tensor([float(n_env_steps_b)], dtype=torch.float64, device='cuda')
            if world > 1:
                dist.all_reduce(tb_t, op=dist.ReduceOp.MAX)
                dist.all_reduce(nb_t, op=dist.ReduceOp.SUM)
            batched['device_gnn_policy'] = {
                'value': float(nb_t[0]) / float(tb_t[0]), 'unit': UNIT, 'ms_per_step': float(tb_t[0]) / K_pol * 1e3,
                'policy': 'GNNPolicy (gnn.yaml: 2 MeanPool rounds, msg 32, hidden 64, read-out [256]), random weights, categorical sampling',
                'trajectory_bytes_per_segment': int(sum(v.nbytes for k_, v in traj.items() if k_ != 'live')),
                'host_decisions': not benv._device_decides_everything}
            pol.close(); benv.close()
        except Exception as ex:
            batched['device_gnn_policy'] = {'error': repr(ex)[:300]}
        batched['what'] = ('RampJobPartitioningEnvironment.step for every episode through the batched gym-like surface (ddls_b200/batched.py), '
                           'host policy (random valid degree from the action mask), actions in and reward / done / observation out as host '
                           'arrays every step; env-steps of episodes that are not done are counted.  device: decision and bookkeeping as '
                           'ramp_env_* kernels; host: the same in numpy + native C++ with caches; device_gnn_policy: the device environment driven by the '
                           'GNN policy kernels (DeviceGNNPolicy.collect: every decision recorded on the device, one read-back of the whole '
                           'trajectory per segment), wall clock over whole segments including resets')

    if rank == 0:
        peak, peak_src = measured_peaks()
        la_ms = kt['total_ms']
        achieved = (kt['algorithmic_bytes'] / 1e9) / (la_ms / 1e3) if la_ms > 0 else 0.0
        prof = ncu_profile_summary()
        n_launch = max(kt['launches'], 1)
        sm_mhz = (clocks or {}).get('sm_mhz') or 1965.0
        roofline = {
            'bound': 'hbm', 'kernel': 'ramp_lookahead_thread_kernel', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
            'frac': achieved / peak if peak else None, 'peak_source': peak_src,
            'definition': 'SURVEY 8d: sum over executed lookaheads of 20 N + 19 E + 12 T + 24 bytes of the LOWERED job handed to '
                          'ramp_register_template, / CUDA-event time of the lookahead launches (bucket + thread kernel) of every step',
            # what the kernel really touches: the symmetry quotient of each job (ramp_quotient.cpp), same formula on its sizes
            'achieved_on_quotient': (kt.get('quotient_bytes', 0) / 1e9) / (la_ms / 1e3) if la_ms > 0 else 0.0,
            'quotient_bytes_per_launch': kt.get('quotient_bytes', 0) / n_launch,
            'traffic': prof.get('dram_bytes_per_launch'), 'traffic_source': prof.get('source'),
            'kernel_ms_per_launch': la_ms / n_launch, 'kernel_launches': kt['launches'],
            'lookaheads': kt['work_items'], 'kernel_share_of_step': la_ms / elapsed_ms if elapsed_ms else None,
            'algorithmic_bytes_per_launch': kt['algorithmic_bytes'] / n_launch,
            # the kernel is bound by the latency of dependent instructions of ONE thread per lookahead, not by bandwidth:
            # warp instructions issued per second against the SM sub-partitions' issue slots (148 x 4 per cycle)
            'issue_slots': {'warp_inst_per_lookahead': prof.get('warp_inst_per_lookahead'),
                            'achieved_warp_inst_per_s': (prof.get('warp_inst_per_lookahead') or 0) * kt['work_items'] / 32.0 / (la_ms / 1e3) if la_ms > 0 else None,
                            'peak_warp_inst_per_s': 148 * 4 * sm_mhz * 1e6, 'source': prof.get('source'),
                            'note': '32 lookaheads share one warp: warp instructions = per-lookahead instructions x lookaheads / 32'}}
        if roofline['issue_slots']['achieved_warp_inst_per_s']:
            roofline['issue_slots']['frac'] = roofline['issue_slots']['achieved_warp_inst_per_s'] / roofline['issue_slots']['peak_warp_inst_per_s']
        # end to end = the call a user makes.  Preferred: the batched gym-like surface on the device
        # (DeviceRampJobPartitioningEnvironment.step(actions[B]) -> obs, reward, done: actions host -> device, observation / reward /
        # done device -> host through page-locked arrays every step, placement + lowering lookup + rewards + observation inside).
        # Also reported: one level down, the C-ABI call ramp_step_host with pre-lowered action rows (round 1's e2e).
        e2e_engine = {'value': e2e_value, 'unit': UNIT, 'api': 'ramp_step_host (C ABI, pre-lowered action rows)',
                      'h2d_bytes_per_step': int(B * engine.ACTION_DTYPE.itemsize + (arrivals.nbytes / L)),
                      'd2h_bytes_per_step': int(B * engine.STEP_STATS_LEN * 8)}
        if batched and isinstance(batched.get('device'), dict) and 'value' in batched['device']:
            n_act = 17
            e2e_line = {'value': batched['device']['value'], 'unit': UNIT,
                        'api': 'ddls_b200.batched.DeviceRampJobPartitioningEnvironment.step(actions) (RJPE.step per episode; host policy: random valid degree)',
                        'h2d_bytes_per_step': int(B * 4), 'd2h_bytes_per_step': int(B * (8 + 1 + 4 + 44 + n_act) + 20),
                        'ms_per_step': batched['device']['ms_per_step']}
        else:
            e2e_line = dict(e2e_engine)
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': elapsed_ms / K, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args, cfg, wl.templates, world, B),
            'trace_mb_per_step': _trace_mb(kt), 'gather_every_steps': gather_every if world > 1 else None,
            'e2e': e2e_line,
            'e2e_engine': e2e_engine,
            'gpu_launches': int(launches),
            'roofline': roofline,
            'memo': {'lookups': memo['lookups'], 'hits': memo['hits'],
                     'hit_rate': memo['hits'] / memo['lookups'] if memo['lookups'] else None},
            'clocks': clocks, 'wall_ms_per_step': wall_ms / K,
            'cluster_steps': {'per_env_step': cluster_steps_per_env_step, 'value': value * cluster_steps_per_env_step,
                              'e2e': e2e_value * cluster_steps_per_env_step, 'unit': 'RampClusterEnvironment.step calls/s'},
            'memo_shared': shared,
            'batched_env': batched,
        }
        if args.config == 'cfg3-resnet50-64w':
            line['python_reference'] = python_reference_note()
            line['template_expansion'] = template_expansion_note()
        if not args.no_cpu_baseline and world == 1:
            line['cpu_baseline'] = cpu_baseline(args, wl)
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def python_reference_note():
    """The unmodified Python reference cannot run on the GPU box; its speed on this config's job was measured once per
    partition degree in the build container when the full-size golden fixtures were generated (oracle/gen_golden.py) and
    travels in the fixtures.  The bench draws the four degrees uniformly, so the mean wall time per env-step is reported."""
    walls = {}
    try:
        for deg in (2, 4, 8, 16):
            d = np.load(os.path.join(ROOT, 'tests', 'golden', f'resnet64_deg{deg}_full.npz'))
            walls[deg] = float(d['meta_reference_wall_s']) / max(int(d['meta_n_env_steps']), 1)
        mean = sum(walls.values()) / len(walls)
        return {'value': 1.0 / mean, 'unit': UNIT, 'cores': 1, 'seconds_per_env_step_by_degree': walls,
                'source': 'tests/golden/resnet64_deg{2,4,8,16}_full.npz: RampJobPartitioningEnvironment.step of the unmodified '
                          'reference on a 64-worker RAMP, ResNet-50-like job, one CPU process in the build container; '
                          'informational, not the reference arm'}
    except Exception:
        return None


def template_expansion_note():
    """Host-side secondary (SURVEY 8f-1): the native expansion of this config's job into a lowered job, per partition degree,
    next to the reference's own agents (whole env-step of the unmodified reference, from the fixtures)."""
    try:
        from ddls_b200 import synth
        from ddls_b200.expand import expand_template
        from ddls_b200.template_builder import RampShape
        g, shape, out = synth.resnet_like_graph(), RampShape(4, 4, 4), {}
        for deg in (2, 4, 8, 16):
            expand_template(g, deg, shape, run_times='reference')
            t0 = time.perf_counter()
            for _ in range(3):
                expand_template(g, deg, shape, run_times='reference')
            out[deg] = (time.perf_counter() - t0) / 3 * 1e3
        ref = python_reference_note() or {}
        return {'native_ms_by_degree': out, 'reference_env_step_s_by_degree': ref.get('seconds_per_env_step_by_degree'),
                'what': 'ramp_expand_template (host C++; partition + dep run times + SRPT priorities + channels -> lowered job, '
                        'bit-identical to the reference pipeline up to hash-ordered priority ties, tests/test_expand_native.py)'}
    except Exception as ex:
        return {'error': str(ex)[:200]}


def _trace_mb(kt):
    # 12 bytes per tick per executed lookahead: (algorithmic bytes - quotient bytes) cancels the per-template part only if the
    # templates were equal, so take the tick term from the quotient accounting: quotient = 20 N' + 19 E' + 24 + 12 T
    return 12.0 * 1400 * kt['work_items'] / max(kt['launches'], 1) / 1e6


def cpu_baseline(args, wl_gpu):
    """Oracle port timed on this box's usable host cores on a bounded sample of the same workload (~10 s of CPU work); the
    unmodified Python reference is timed by the reference arm (`bench.py --impl reference`)."""
    cores = usable_cores()
    out = port_throughput(args, cores['used'], budget_s=10.0)
    out['host_cores'] = cores
    return out


def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference_arm(args, rank, world)
    else:
        run_b200_arm(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
