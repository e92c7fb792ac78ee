"""TEST INFRASTRUCTURE -- ctypes binding of the CPU oracle (oracle/ramp_oracle.c).

Only tests/, bench.py's cpu_baseline / ``--impl reference`` legs and
``__graft_entry__.smoke()`` may import this module.  The product never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, 'libramp_oracle.so')

STEP_STATS = [
    'step_counter', 'step_start_time', 'step_end_time', 'step_time', 'num_jobs_completed', 'num_jobs_arrived',
    'num_jobs_blocked', 'job_queue_length', 'mean_num_jobs_running', 'mean_num_mounted_workers',
    'mean_num_mounted_channels', 'mean_compute_overhead_frac', 'mean_communication_overhead_frac',
    'compute_info_processed', 'dep_info_processed', 'flow_info_processed', 'cluster_info_processed',
    'demand_compute_info_processed', 'demand_dep_info_processed', 'demand_total_info_processed',
    'mean_compute_throughput', 'mean_dep_throughput', 'mean_flow_throughput', 'mean_cluster_throughput',
    'mean_demand_compute_throughput', 'mean_demand_dep_throughput', 'mean_demand_total_throughput',
    'util_mounted_sum', 'util_cluster_sum', 'num_ticks', 'done', 'lookahead_ran']
SS = {k: i for i, k in enumerate(STEP_STATS)}
STEP_STATS_LEN = len(STEP_STATS)

JS_NOT_ARRIVED, JS_QUEUED, JS_RUNNING, JS_COMPLETED, JS_BLOCKED = range(5)
ORC_OK, ORC_ERR_INFINITE_TICK, ORC_ERR_TRACE_OVERFLOW = 0, 1, 2


class CLoweredJob(C.Structure):
    _fields_ = [('n_ops', C.c_int32), ('n_deps', C.c_int32), ('n_workers', C.c_int32), ('n_channels', C.c_int32),
                ('num_training_steps', C.c_int32), ('model_id', C.c_int32), ('degree', C.c_int32), ('_pad', C.c_int32),
                ('op_cost', C.c_void_p), ('op_prio', C.c_void_p), ('op_worker', C.c_void_p),
                ('op_n_parents', C.c_void_p), ('row_ptr', C.c_void_p), ('dep_dst', C.c_void_p),
                ('dep_run_time', C.c_void_p), ('dep_prio', C.c_void_p), ('dep_channel', C.c_void_p),
                ('dep_is_flow', C.c_void_p)]


class CLookaheadResult(C.Structure):
    _fields_ = [('jct', C.c_double), ('comm', C.c_double), ('comp', C.c_double),
                ('n_ticks', C.c_int32), ('status', C.c_int32)]


class CArrival(C.Structure):
    _fields_ = [('interarrival', C.c_double), ('orig_op_mem', C.c_double), ('orig_dep_size', C.c_double)]


class CMount(C.Structure):
    _fields_ = [('max_acceptable_jct', C.c_double), ('part_op_mem', C.c_double), ('part_dep_size', C.c_double),
                ('flow_size', C.c_double), ('n_mounted_workers', C.c_int32), ('n_mounted_channels', C.c_int32)]


class CJobRecord(C.Structure):
    _fields_ = [('status', C.c_int32), ('event_seq', C.c_int32), ('time_arrived', C.c_double),
                ('time_started', C.c_double), ('time_completed', C.c_double), ('jct', C.c_double),
                ('comm', C.c_double), ('comp', C.c_double), ('util', C.c_double)]


JOB_RECORD_DTYPE = np.dtype([('status', np.int32), ('event_seq', np.int32), ('time_arrived', np.float64),
                             ('time_started', np.float64), ('time_completed', np.float64), ('jct', np.float64),
                             ('comm', np.float64), ('comp', np.float64), ('util', np.float64)])
ARRIVAL_DTYPE = np.dtype([('interarrival', np.float64), ('orig_op_mem', np.float64), ('orig_dep_size', np.float64)])
MOUNT_DTYPE = np.dtype([('max_acceptable_jct', np.float64), ('part_op_mem', np.float64), ('part_dep_size', np.float64),
                        ('flow_size', np.float64), ('n_mounted_workers', np.int32), ('n_mounted_channels', np.int32)])

_lib = None


def build(force=False):
    """Compiles oracle/libramp_oracle.so from the C restatement (gcc, -ffp-contract=off)."""
    srcs = [os.path.join(_HERE, f) for f in ('ramp_oracle.c', 'ramp_oracle_batch.c', 'ramp_oracle.h', 'Makefile')]
    if (not force and os.path.exists(_LIB_PATH)
            and all(os.path.getmtime(_LIB_PATH) >= os.path.getmtime(s) for s in srcs)):
        return _LIB_PATH
    subprocess.check_call(['make', '-C', _HERE, '-s', '-B'])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        L.orc_run_lookahead.restype = C.c_int
        L.orc_run_lookahead.argtypes = [C.POINTER(CLoweredJob), C.c_void_p, C.c_void_p, C.c_int32,
                                        C.POINTER(CLookaheadResult)]
        L.orc_utilisation.restype = C.c_double
        L.orc_utilisation.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double]
        L.orc_env_create.restype = C.c_void_p
        L.orc_env_create.argtypes = [C.c_int32] * 6 + [C.c_double]
        L.orc_env_destroy.argtypes = [C.c_void_p]
        L.orc_env_reset.restype = C.c_int
        L.orc_env_reset.argtypes = [C.c_void_p, C.c_double, C.c_int32, C.c_void_p, C.c_int32]
        L.orc_env_step.restype = C.c_int
        L.orc_env_step.argtypes = [C.c_void_p, C.POINTER(CLoweredJob), C.POINTER(CMount), C.c_void_p]
        L.orc_env_set_arrival.restype = C.c_int
        L.orc_env_set_arrival.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_env_set_job_count.restype = C.c_int
        L.orc_env_set_job_count.argtypes = [C.c_void_p, C.c_int32]
        L.orc_env_tick_lists.restype = C.c_int32
        L.orc_env_tick_lists.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        L.orc_env_queued_job.restype = C.c_int32
        L.orc_env_queued_job.argtypes = [C.c_void_p]
        L.orc_env_num_jobs_arrived.restype = C.c_int32
        L.orc_env_num_jobs_arrived.argtypes = [C.c_void_p]
        L.orc_env_time.restype = C.c_double
        L.orc_env_time.argtypes = [C.c_void_p]
        L.orc_env_mean_load_rate.restype = C.c_double
        L.orc_env_mean_load_rate.argtypes = [C.c_void_p]
        L.orc_env_job_records.restype = C.c_void_p
        L.orc_env_job_records.argtypes = [C.c_void_p]
        L.orc_env_last_trace.restype = C.c_int32
        L.orc_env_last_trace.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
        L.orc_run_lookahead_batch.restype = C.c_int
        L.orc_run_lookahead_batch.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]
        L.orc_run_scripted_batch.restype = C.c_int
        L.orc_run_scripted_batch.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_int32, C.c_double, C.c_int32, C.c_int32, C.c_int32,
                                             C.c_void_p, C.c_void_p, C.c_int32]
        L.orc_run_scripted_rjpe_batch.restype = C.c_int
        L.orc_run_scripted_rjpe_batch.argtypes = L.orc_run_scripted_batch.argtypes
        L.orc_run_scripted_rjpe_batch_ex.restype = C.c_int
        L.orc_run_scripted_rjpe_batch_ex.argtypes = L.orc_run_scripted_batch.argtypes[:-1] + [C.c_void_p, C.c_int32]
        _lib = L
    return _lib


def to_c(job):
    """LoweredJob -> CLoweredJob (keeps the numpy arrays alive via the returned struct)."""
    cj = CLoweredJob(job.n_ops, job.n_deps, job.n_workers, job.n_channels, job.num_training_steps,
                     job.model_id, job.degree, 0,
                     job.op_cost.ctypes.data, job.op_prio.ctypes.data, job.op_worker.ctypes.data,
                     job.op_n_parents.ctypes.data, job.row_ptr.ctypes.data, job.dep_dst.ctypes.data,
                     job.dep_run_time.ctypes.data, job.dep_prio.ctypes.data, job.dep_channel.ctypes.data,
                     job.dep_is_flow.ctypes.data)
    cj._keep = job
    return cj


def to_c_mount(m):
    return CMount(m.max_acceptable_jct, m.part_op_mem, m.part_dep_size, m.flow_size,
                  m.n_mounted_workers, m.n_mounted_channels)


def run_lookahead(job, trace_cap=None):
    """Returns dict(jct, comm, comp, n_ticks, status, trace_n_active, trace_tick)."""
    cap = (job.n_ops + job.n_deps + 1) if trace_cap is None else trace_cap
    tn = np.zeros(max(cap, 1), dtype=np.int32)
    tt = np.zeros(max(cap, 1), dtype=np.float64)
    res = CLookaheadResult()
    cj = to_c(job)
    lib().orc_run_lookahead(C.byref(cj), tn.ctypes.data, tt.ctypes.data, cap, C.byref(res))
    T = min(res.n_ticks, cap)
    return dict(jct=res.jct, comm=res.comm, comp=res.comp, n_ticks=res.n_ticks, status=res.status,
                trace_n_active=tn[:T].copy(), trace_tick=tt[:T].copy())


def utilisation(trace_n_active, trace_tick, n_mounted_workers, jct):
    tn = np.ascontiguousarray(trace_n_active, dtype=np.int32)
    tt = np.ascontiguousarray(trace_tick, dtype=np.float64)
    return lib().orc_utilisation(tn.ctypes.data, tt.ctypes.data, len(tn), n_mounted_workers, jct)


def run_scripted(templates, script_tid, script_mount, arrivals, n_workers, n_models, n_threads=None,
                 max_simulation_run_time=float('inf')):
    """B independent scripted episodes of L RampJobPartitioningEnvironment.step calls each (RJPE:300-420), one oracle env per
    episode, spread over ``n_threads`` host threads.  Env-step s of episode b mounts ``templates[script_tid[b, s]]`` with the
    mount scalars ``script_mount[b, s]`` (MOUNT_DTYPE) when a job is queued, else (or when the id is -1) is Action(); then
    Action() steps follow until a job is queued or the episode is done.

    Returns (stats [B, L, STEP_STATS_LEN] f64: the action step's statistics with `done` after the whole env-step,
    records [B, J] JOB_RECORD_DTYPE, cluster_steps [B, L] int32: RampClusterEnvironment.step calls of each env-step)."""
    tid = np.ascontiguousarray(script_tid, dtype=np.int32)
    B, L = tid.shape
    mount = np.ascontiguousarray(script_mount, dtype=MOUNT_DTYPE)
    arr = np.ascontiguousarray(arrivals, dtype=ARRIVAL_DTYPE)
    assert mount.shape == (B, L) and arr.ndim == 2 and arr.shape[0] == B
    J = arr.shape[1]
    keep = [to_c(t) for t in templates]                      # the structs point into the templates' arrays
    ctemps = (CLoweredJob * max(len(keep), 1))(*keep)
    stats = np.zeros((B, L, STEP_STATS_LEN), dtype=np.float64)
    records = np.zeros((B, J), dtype=JOB_RECORD_DTYPE)
    ncs = np.zeros((B, L), dtype=np.int32)
    if n_threads is None:
        n_threads = len(os.sched_getaffinity(0))
    rc = lib().orc_run_scripted_rjpe_batch_ex(ctemps, len(keep), B, L, tid.ctypes.data, mount.ctypes.data, arr.ctypes.data, J,
                                              float(max_simulation_run_time), int(n_workers), int(n_models), 1025,
                                              stats.ctypes.data, records.ctypes.data, ncs.ctypes.data, int(n_threads))
    if rc != 0:
        raise Exception(f'orc_run_scripted_rjpe_batch_ex failed with status {rc}')
    del keep
    return stats, records, ncs


class OracleEnv:
    """Episode-level oracle: RampClusterEnvironment.reset()/step() on lowered jobs."""

    def __init__(self, n_cluster_workers, max_jobs, memo_models=8, memo_degrees=1025, machine_epsilon=1e-7):
        self.max_jobs = max_jobs
        self._h = lib().orc_env_create(n_cluster_workers, max(n_cluster_workers, 1), max_jobs,
                                       memo_models, memo_degrees, 0, machine_epsilon)

    def __del__(self):
        if getattr(self, '_h', None):
            lib().orc_env_destroy(self._h)
            self._h = None

    def reset(self, arrivals, max_simulation_run_time=float('inf'), job_queue_capacity=10):
        arr = np.ascontiguousarray(arrivals, dtype=ARRIVAL_DTYPE)
        self._n_jobs = len(arr)
        rc = lib().orc_env_reset(self._h, max_simulation_run_time, job_queue_capacity, arr.ctypes.data, len(arr))
        if rc != 0:
            raise Exception(f'orc_env_reset failed with status {rc}')

    def set_arrival(self, k, row):
        r = np.ascontiguousarray(row, dtype=ARRIVAL_DTYPE).reshape(1)
        if lib().orc_env_set_arrival(self._h, k, r.ctypes.data) != 0:
            raise Exception('orc_env_set_arrival failed')
        self._n_jobs = max(self._n_jobs, k + 1)

    def set_job_count(self, n):
        if lib().orc_env_set_job_count(self._h, n) != 0:
            raise Exception('orc_env_set_job_count failed')

    def tick_lists(self):
        """The last step's step_stats['mean_mounted_worker_utilisation_frac'] / ['mean_cluster_worker_utilisation_frac'] (RCE:989-994)."""
        n = lib().orc_env_tick_lists(self._h, None, None, 0)
        a, b = np.zeros(max(n, 1)), np.zeros(max(n, 1))
        lib().orc_env_tick_lists(self._h, a.ctypes.data, b.ctypes.data, n)
        return a[:n], b[:n]

    def step(self, job=None):
        stats = np.zeros(STEP_STATS_LEN, dtype=np.float64)
        if job is None:
            rc = lib().orc_env_step(self._h, None, None, stats.ctypes.data)
        else:
            cj, cm = to_c(job), to_c_mount(job.mount)
            rc = lib().orc_env_step(self._h, C.byref(cj), C.byref(cm), stats.ctypes.data)
        if rc != 0:
            raise Exception(f'orc_env_step failed with status {rc}')
        return stats

    @property
    def queued_job(self):
        return lib().orc_env_queued_job(self._h)

    @property
    def time(self):
        return lib().orc_env_time(self._h)

    @property
    def mean_load_rate(self):
        return lib().orc_env_mean_load_rate(self._h)

    def job_records(self):
        ptr = lib().orc_env_job_records(self._h)
        buf = (C.c_char * (JOB_RECORD_DTYPE.itemsize * self._n_jobs)).from_address(ptr)
        return np.frombuffer(buf, dtype=JOB_RECORD_DTYPE).copy()

    def last_trace(self):
        pn, pt = C.c_void_p(), C.c_void_p()
        T = lib().orc_env_last_trace(self._h, C.byref(pn), C.byref(pt))
        if T == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.float64)
        tn = np.frombuffer((C.c_char * (4 * T)).from_address(pn.value), dtype=np.int32).copy()
        tt = np.frombuffer((C.c_char * (8 * T)).from_address(pt.value), dtype=np.float64).copy()
        return tn, tt
