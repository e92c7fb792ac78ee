"""TEST INFRASTRUCTURE: replays a recorded drop-in session on ``ddls_b200.host.RampClusterEnvironment``.

A session (tests/golden/dropin/<case>.npz, written by ``tests/ref_dropin_driver.py --record``) holds everything the
reference's RampJobPartitioningEnvironment and agents handed to the drop-in cluster environment in one seeded episode:
the jobs and inter-arrival gaps its job generator produced, the answers of ``len(jobs_generator)``, and for every
``step`` the Action -- as the lowered job it lowers to, its global worker / channel ids and mount scalars.  The replay
rebuilds reference-shaped Job and Action objects from it (ddls_b200/host/synthetic.py), drives a fresh drop-in through
the same calls and reports what the drop-in produced, in the form the reference-side driver reports it.

    PYTHONHASHSEED=0 python tests/dropin_replay.py <case> [--fake-engine]

--fake-engine answers the engine calls with the CPU oracle (tests/fake_engine.py); without it the CUDA engine is used."""
import copy
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

SESSION_DIR = os.path.join(HERE, 'golden', 'dropin')
DEVICE_TYPE = 'A100'
ES_SCALARS = ('episode_end_time', 'mean_load_rate', 'blocking_rate', 'acceptance_rate', 'compute_info_processed', 'dep_info_processed',
              'flow_info_processed', 'cluster_info_processed', 'mean_compute_throughput', 'mean_cluster_throughput',
              'mean_compute_overhead_frac', 'mean_communication_overhead_frac', 'mean_num_jobs_running', 'mean_num_mounted_workers')
ES_LISTS = ('job_completion_time', 'job_completion_time_speedup', 'job_communication_overhead_time', 'job_computation_overhead_time',
            'jobs_completed_mean_mounted_worker_utilisation_frac', 'jobs_completed_num_mounted_workers',
            'jobs_completed_num_mounted_channels', 'jobs_completed_max_acceptable_job_completion_time',
            'jobs_blocked_max_acceptable_job_completion_time')


def cluster_result(cluster, n_env_steps, actions, is_dropin, using_reference_classes):
    """What one episode left in a cluster environment (the reference's or the drop-in), as plain JSON-able data."""
    es = cluster.episode_stats
    out = {'n_env_steps': int(n_env_steps), 'actions': [int(a) for a in actions], 'using_reference_classes': bool(using_reference_classes),
           'n_cluster_steps': len(cluster.steps_log['step_end_time']),
           'completed_job_idxs': [int(k) for k in cluster.jobs_completed.keys()],
           'blocked_job_idxs': [int(k) for k in cluster.jobs_blocked.keys()],
           'steps_log': {k: [float(x) for x in cluster.steps_log[k]] for k in
                         ('step_start_time', 'step_end_time', 'num_jobs_completed', 'num_jobs_arrived', 'num_jobs_blocked',
                          'mean_num_jobs_running', 'mean_compute_overhead_frac', 'mean_communication_overhead_frac',
                          'compute_info_processed', 'mean_cluster_throughput')},
           # the two step statistics the reference leaves as per-tick lists (RCE:989-994)
           'tick_lists': {k: [[float(x) for x in step] for step in cluster.steps_log[k]] for k in
                          ('mean_mounted_worker_utilisation_frac', 'mean_cluster_worker_utilisation_frac')}}
    for k in ('num_jobs_arrived', 'num_jobs_completed', 'num_jobs_blocked'):
        out[k] = int(es[k])
    for k in ES_SCALARS:
        out[k] = float(es[k])
    for k in ES_LISTS:
        out[k] = [float(x) for x in es[k]]
    memo = cluster.job_model_to_max_num_partitions_to_init_details
    out['is_dropin'] = bool(is_dropin)
    out['last_step_stats'] = {k: float(cluster.step_stats[k]) for k in ('num_jobs_blocked', 'num_jobs_completed', 'num_jobs_arrived', 'step_end_time')}
    out['init_details_memo_keys'] = sorted([str(m), int(p)] for m in memo for p in memo[m])
    return out


class _ReplayGenerator:
    """The job generator as the drop-in saw it: the recorded jobs and gaps in draw order, the recorded len() answers."""

    def __init__(self, jobs, gaps, lens):
        self._jobs, self._gaps, self._lens = list(jobs), list(gaps), [int(n) for n in lens]
        self.jobs_params = {}

    def __len__(self):
        return self._lens.pop(0)

    def sample_job(self):
        return self._jobs.pop(0)

    def sample_interarrival_time(self, size=None):
        return self._gaps.pop(0)


def _reset_job(job, details, job_total_operation_memory_cost=None, job_total_dependency_size=None, init_job_immutable_details=None):
    """The part of the reference's Job.reset_job the cluster environment reads back: the job totals, the immutable details
    it memoises per (model, max partition degree), and the lookahead's details."""
    if job_total_operation_memory_cost is not None:
        job.job_total_operation_memory_cost = job_total_operation_memory_cost
    if job_total_dependency_size is not None:
        job.job_total_dependency_size = job_total_dependency_size
    job.init_job_immutable_details = init_job_immutable_details if init_job_immutable_details is not None else {'model': job.details['model']}
    job.details.update(details)


def _strings(d, key, s):
    ptr = d[key + '_ptr']
    return [str(x) for x in d[key][ptr[s]:ptr[s + 1]]]


def load_session(case):
    from golden_io import Golden
    from ddls_b200.lowered import LoweredJob
    d = np.load(os.path.join(SESSION_DIR, f'{case}.npz'))
    base = str(d['base'])
    templates = list(Golden(base).templates) if base else []
    templates += [LoweredJob.from_npz_dict(d, prefix=f'x{i}_') for i in range(int(d['n_extra']))]
    return d, templates


def replay(case, fake):
    from ddls_b200.host import synthetic
    from ddls_b200.lowered import MountScalars
    import ddls_b200.host.cluster as host_cluster
    from ddls_b200 import host
    if fake:
        from fake_engine import FakeEngine
        host_cluster._engine.RampEngine = FakeEngine
    d, templates = load_session(case)
    c, r, s = (int(x) for x in d['shape'])
    env = host.RampClusterEnvironment(
        topology_config={'type': 'ramp', 'kwargs': {'num_communication_groups': c, 'num_racks_per_communication_group': r,
                                                    'num_servers_per_rack': s, 'num_channels': 1, 'total_node_bandwidth': 1.6e12,
                                                    'intra_gpu_propagation_latency': 50e-9, 'worker_io_latency': 100e-9}},
        node_config={'type_1': {'num_nodes': c * r * s, 'workers_config': [{'num_workers': 1, 'worker': host.A100}]}},
        suppress_warnings=True)
    jobs = []
    for k, (gap, op_mem, dep_size, seq_time, max_jct, frac, n_steps) in enumerate(d['draw_f']):
        job = synthetic.build_original_job(int(d['draw_job_id'][k]), str(d['draw_model'][k]), float(op_mem), float(dep_size),
                                           float(frac), float(seq_time), int(n_steps))
        job.details['max_acceptable_job_completion_time'] = {DEVICE_TYPE: float(max_jct)}
        jobs.append(job)
    max_sim_time, queue_capacity = d['reset']
    env.reset(_ReplayGenerator(jobs, [float(g) for g in d['draw_f'][:, 0]], d['gen_len']),
              max_simulation_run_time=float(max_sim_time), job_queue_capacity=int(queue_capacity))
    for st in range(len(d['step_tid'])):
        tid = int(d['step_tid'][st])
        if tid < 0:
            action = synthetic.SyntheticAction()
        else:
            job_id = int(d['step_job_id'][st])
            queued = env.job_queue.jobs[job_id]
            lj = copy.copy(templates[tid])
            m = d['step_mount'][st]
            lj.mount = MountScalars(float(m[0]), float(m[1]), float(m[2]), float(m[3]), int(m[4]), int(m[5]))
            action, pjob = synthetic.build_action(lj, queued, env, worker_ids=_strings(d, 'step_workers', st),
                                                  channel_ids=_strings(d, 'step_channels', st))
            pjob.details['job_sequential_completion_time'] = {DEVICE_TYPE: float(d['step_seq_time'][st])}
            pjob.reset_job = lambda job=pjob, **kw: _reset_job(job, **kw)
            action.actions['op_partition'].job_id_to_partitioned_computation_graph = {job_id: pjob.computation_graph}
        env.step(action)
    assert env.is_done()
    return cluster_result(env, int(d['n_env_steps']), d['actions'], is_dropin=True, using_reference_classes=host.USING_REFERENCE_CLASSES)


if __name__ == '__main__':
    out = replay(sys.argv[1], fake='--fake-engine' in sys.argv)
    print('RESULT ' + json.dumps(out), flush=True)
