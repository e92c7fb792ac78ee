"""TEST INFRASTRUCTURE: the subset of ``ddls_b200.engine.RampEngine`` the drop-in cluster environment uses, answered by the
CPU oracle (oracle/ramp_oracle.c).  Lets the host-side logic of ``ddls_b200.host.RampClusterEnvironment`` be driven the way
the reference's own RampJobPartitioningEnvironment and agents drive it where there is no GPU (tests/test_reference_dropin.py);
the same test runs against the CUDA engine under ``-m gpu``.  Never imported by the product."""
import copy

import numpy as np

from ddls_b200 import engine as _engine
from ddls_b200.lowered import MountScalars
from oracle import oracle


class FakeEngine:
    def __init__(self, n_episodes, n_cluster_workers, max_jobs, device=0, memo_mode=0, job_queue_capacity=10,
                 machine_epsilon=1e-7, max_simulation_run_time=float('inf'), **_):
        assert n_episodes == 1 and memo_mode == _engine.MEMO_REFERENCE
        self.n_episodes, self.max_jobs = 1, max_jobs
        self._env = oracle.OracleEnv(n_cluster_workers, max_jobs=max_jobs, memo_models=64, machine_epsilon=machine_epsilon)
        self._limits = (max_simulation_run_time, job_queue_capacity)
        self._templates = []
        self._done = 0.0

    def close(self):
        self._env = None

    def register_template(self, job):
        job.canonicalise()
        self._templates.append(job)
        return len(self._templates) - 1

    def set_limits(self, max_simulation_run_time=float('inf'), job_queue_capacity=10):
        self._limits = (max_simulation_run_time, job_queue_capacity)

    def reset(self, arrivals):
        arr = np.ascontiguousarray(arrivals, dtype=_engine.ARRIVAL_DTYPE)
        self._env.reset(arr[0], max_simulation_run_time=self._limits[0], job_queue_capacity=self._limits[1])
        self._done = 0.0

    def set_arrivals(self, episode, first_job, rows):
        rows = np.ascontiguousarray(rows, dtype=_engine.ARRIVAL_DTYPE).reshape(-1)
        for k, r in enumerate(rows):
            self._env.set_arrival(first_job + k, r)

    def set_job_count(self, episode, n_jobs):
        self._env.set_job_count(n_jobs)

    def make_actions(self):
        a = np.zeros(1, dtype=_engine.ACTION_DTYPE)
        a['template_id'] = -1
        return a

    def episode_state(self):
        out = np.zeros((1, len(_engine.EP_FIELDS)))
        out[0, _engine.EP['time']] = self._env.time
        out[0, _engine.EP['queued_job']] = self._env.queued_job
        out[0, _engine.EP['done']] = self._done
        return out

    def step(self, actions, **_):
        tid = int(actions['template_id'][0])
        job = None
        if tid >= 0:
            job = copy.copy(self._templates[tid])
            a = actions[0]
            job.mount = MountScalars(float(a['max_acceptable_jct']), float(a['part_op_mem']), float(a['part_dep_size']),
                                     float(a['flow_size']), int(a['n_mounted_workers']), int(a['n_mounted_channels']))
        stats = self._env.step(job).reshape(1, -1)
        self._done = float(stats[0, _engine.SS['done']])
        return stats

    def enable_tick_lists(self, cap=256):
        pass                      # the oracle always keeps them

    def tick_lists(self, episode=0):
        return self._env.tick_lists()

    def check_status(self):
        pass                      # OracleEnv.step raises on the same conditions

    def job_records(self):
        rec = self._env.job_records()
        out = np.zeros((1, self.max_jobs), dtype=_engine.JOB_RECORD_DTYPE)
        for f in rec.dtype.names:
            out[0, :len(rec)][f] = rec[f]
        return out
