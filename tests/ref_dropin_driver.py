"""TEST INFRASTRUCTURE: drives the UNMODIFIED reference's RampJobPartitioningEnvironment + heuristic agents with
``ddls_b200.host.RampClusterEnvironment`` swapped in for the reference's cluster environment (the INTEGRATION.md stub:
RJPE:199-206), on one of the seeded golden episodes, and prints what the reference itself recorded for that episode
(tests/golden/<case>.npz) next to what this run produced.

    PYTHONHASHSEED=0 python tests/ref_dropin_driver.py <case> [--fake-engine] [--reference-cluster] [--record PATH]

--fake-engine answers the engine calls with the CPU oracle (tests/fake_engine.py) so the host logic can be checked
without a GPU; without it the CUDA engine is used (needs cuda:0).  --reference-cluster runs the reference's own cluster
environment instead of the drop-in.  Needs the reference checkout, so the suite does not run it; it regenerates the
fixtures the suite replays:

    PYTHONHASHSEED=0 python tests/ref_dropin_driver.py <case> --fake-engine --record tests/golden/dropin/<case>.npz
    PYTHONHASHSEED=0 python tests/ref_dropin_driver.py <case> --fake-engine --reference-cluster   # RESULT line ->
                                                                              # tests/golden/dropin/<case>_reference.json"""
import json
import os
import random
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


# The reference lists its job files with an UNSORTED glob (jobs_generator.py:96), so which file is "job type 0" depends on the
# file system's directory order.  These are the orders of the container the golden fixtures were generated in; the driver pins
# them so that the seeded episodes are the same episodes on every machine.
FILE_ORDER = {'mixed16': ['res2.txt', 'chain5.txt', 'tfm1.txt'], 'mixed64_busy': ['tfm1b.txt', 'chain4.txt', 'res1.txt'],
              'mix128_exp': ['resnet50_like.txt', 'gpt2_small_like.txt']}

EXTRA_CASES = {
    # a generator that never runs dry (the reference's default 'remove_and_repeat' sampling, heuristic_config.yaml:126): the
    # episode ends on max_simulation_run_time, arrivals keep coming until then
    'chain8_repeat': dict(base='chain8', sampling_mode='remove_and_repeat', max_sim_time=9500.0, n_jobs=3),
    'res16_repeat': dict(base='res16_flood', sampling_mode='remove_and_repeat', max_sim_time=700.0, n_jobs=2),
}


class _RecordingGenerator:
    """Wraps the reference's JobsGenerator: every job, gap and len() answer the drop-in receives is recorded."""

    def __init__(self, gen, rec):
        self._gen, self._rec = gen, rec

    def __len__(self):
        n = len(self._gen)
        self._rec.gen_len.append(n)
        return n

    def sample_job(self):
        job = self._gen.sample_job()
        self._rec.draws.append(job)
        return job

    def sample_interarrival_time(self, size=None):
        gap = self._gen.sample_interarrival_time(size=size)
        self._rec.gaps.append(float(gap))
        return gap

    def __getattr__(self, name):
        return getattr(self._gen, name)


class SessionRecorder:
    """Records what the reference hands to the drop-in cluster environment in the last episode (reset onwards) as a
    session for tests/dropin_replay.py: jobs and gaps drawn, len(jobs_generator) answers, and per step the lowered Action
    with its global worker / channel ids.  Lowered jobs already in the case's golden fixture are referred to by index."""

    def __init__(self, base, shape):
        from ddls_b200.lowering import ModelRegistry
        from golden_io import Golden
        self.base, self.shape = base, shape
        self.models = ModelRegistry()
        self.known = list(Golden(base).templates) if base else []
        self.extra = []
        self._clear()

    def _clear(self):
        self.gen_len, self.draws, self.gaps, self.steps, self.reset_args = [], [], [], [], None

    def _tid(self, lj):
        key = (lj.fingerprint(), lj.degree)
        for i, t in enumerate(self.known + self.extra):
            if (t.fingerprint(), t.degree) == key:
                return i
        self.extra.append(lj)
        return len(self.known) + len(self.extra) - 1

    def install(self, cls):
        from ddls_b200.lowering import lower_job
        rec, orig_reset, orig_step = self, cls.reset, cls.step

        def reset(cluster, jobs_config, max_simulation_run_time=float('inf'), job_queue_capacity=10, seed=None, verbose=False):
            if isinstance(jobs_config, dict):
                from ddls.demands.jobs.jobs_generator import JobsGenerator
                jobs_config = JobsGenerator(**jobs_config)
            rec._clear()
            rec.reset_args = (float(max_simulation_run_time), int(job_queue_capacity))
            return orig_reset(cluster, _RecordingGenerator(jobs_config, rec), max_simulation_run_time, job_queue_capacity, seed, verbose)

        def step(cluster, action, verbose=False):
            entry = {'tid': -1}
            job_ids = list(action.job_ids)
            if len(job_ids) == 1:
                lj = lower_job(cluster, action, job_ids[0], rec.models)        # before the step mounts the job
                pjob = action.actions['op_partition'].partitioned_jobs[job_ids[0]]
                entry = {'tid': rec._tid(lj), 'job_id': int(job_ids[0]), 'mount': lj.mount, 'workers': list(lj.worker_ids),
                         'channels': list(lj.channel_ids), 'seq_time': float(pjob.details['job_sequential_completion_time']['A100'])}
            rec.steps.append(entry)
            return orig_step(cluster, action, verbose=verbose)

        cls.reset, cls.step = reset, step

    def save(self, path, n_env_steps, actions):
        out = {'base': np.array(self.base), 'shape': np.array(self.shape, dtype=np.int64), 'reset': np.array(self.reset_args),
               'gen_len': np.array(self.gen_len, dtype=np.int64), 'n_env_steps': np.array(n_env_steps),
               'actions': np.array(actions, dtype=np.int64)}
        assert len(self.gaps) == len(self.draws)
        out['draw_job_id'] = np.array([int(j.job_id) for j in self.draws], dtype=np.int64)
        out['draw_model'] = np.array([str(j.details['model']) for j in self.draws])
        out['draw_f'] = np.array([[gap, j.original_job.details['job_total_op_memory_cost'], j.original_job.details['job_total_dep_size'],
                                   j.details['job_sequential_completion_time']['A100'], j.details['max_acceptable_job_completion_time']['A100'],
                                   j.max_acceptable_job_completion_time_frac, j.num_training_steps]
                                  for j, gap in zip(self.draws, self.gaps)], dtype=np.float64).reshape(-1, 7)
        out['step_tid'] = np.array([e['tid'] for e in self.steps], dtype=np.int32)
        out['step_job_id'] = np.array([e.get('job_id', -1) for e in self.steps], dtype=np.int64)
        out['step_seq_time'] = np.array([e.get('seq_time', 0.0) for e in self.steps], dtype=np.float64)
        out['step_mount'] = np.array([[e['mount'].max_acceptable_jct, e['mount'].part_op_mem, e['mount'].part_dep_size, e['mount'].flow_size,
                                       e['mount'].n_mounted_workers, e['mount'].n_mounted_channels] if e['tid'] >= 0 else [0.0] * 6
                                      for e in self.steps], dtype=np.float64)
        for key in ('workers', 'channels'):
            lists = [e.get(key, []) for e in self.steps]
            out[f'step_{key}'] = np.array([str(x) for lst in lists for x in lst])
            out[f'step_{key}_ptr'] = np.concatenate([[0], np.cumsum([len(lst) for lst in lists])]).astype(np.int64)
        out['n_extra'] = np.array(len(self.extra))
        for i, lj in enumerate(self.extra):
            out.update(lj.to_npz_dict(prefix=f'x{i}_'))
        os.makedirs(os.path.dirname(path), exist_ok=True)
        np.savez_compressed(path, **out)


def main():
    case = sys.argv[1]
    fake = '--fake-engine' in sys.argv
    use_reference_cluster = '--reference-cluster' in sys.argv      # run the reference's own cluster environment instead
    record_path = sys.argv[sys.argv.index('--record') + 1] if '--record' in sys.argv else None
    from oracle import ref_shim
    ref_shim.install()
    from dropin_replay import cluster_result
    from oracle import gen_golden                     # CASES / make_env / the reference imports (no recording here)
    import ddls.environments.ramp_job_partitioning.ramp_job_partitioning_environment as rjpe_mod
    from ddls.distributions.uniform import Uniform
    from ddls.environments.ramp_job_partitioning.agents.sip_ml import SiPML
    from ddls.environments.ramp_job_partitioning.agents.random import Random
    from ddls.environments.ramp_job_partitioning.agents.acceptable_jct import AcceptableJCT
    import ddls_b200.host.cluster as host_cluster
    from ddls_b200 import host
    if fake:
        from fake_engine import FakeEngine
        host_cluster._engine.RampEngine = FakeEngine
    if not use_reference_cluster:
        rjpe_mod.RampClusterEnvironment = host.RampClusterEnvironment        # the drop-in (RJPE:199-206)

    sampling_mode = 'remove'
    if case in EXTRA_CASES:
        extra = dict(EXTRA_CASES[case])
        spec = dict(gen_golden.CASES[extra.pop('base')])
        sampling_mode = extra.pop('sampling_mode')
        spec.update(extra)
    else:
        spec = gen_golden.CASES[case]
    recorder = None
    if record_path is not None:
        assert not use_reference_cluster
        recorder = SessionRecorder('' if case in EXTRA_CASES else case, spec['shape'])
        recorder.install(host_cluster.RampClusterEnvironment)
    seed = spec['seed']
    np.random.seed(seed)
    random.seed(seed)
    d = tempfile.mkdtemp(prefix='dropin_graphs_')
    for g in spec['graphs']:
        g.write(d)
    if case in FILE_ORDER:
        import ddls.demands.jobs.jobs_generator as jg_mod
        import glob as _glob
        real_glob = _glob.glob

        class _PinnedGlob:
            @staticmethod
            def glob(pattern, *a, **kw):
                found = real_glob(pattern, *a, **kw)
                rank = {n: i for i, n in enumerate(FILE_ORDER[case])}
                return sorted(found, key=lambda pth: rank.get(os.path.basename(pth), len(rank)))
        jg_mod.glob = _PinnedGlob
    env = gen_golden.make_env(d, spec['shape'], spec['n_jobs'], spec['max_partitions'], spec['interarrival'],
                              Uniform(spec['frac'][0], spec['frac'][1], decimals=2), max_sim_time=spec.get('max_sim_time', 1e6),
                              sampling_mode=sampling_mode)
    assert isinstance(env.cluster, host.RampClusterEnvironment) != use_reference_cluster
    np.random.seed(seed)
    random.seed(seed)
    obs = env.reset()
    actor = {'random': Random(), 'sipml': SiPML(spec['max_partitions']), 'acceptable_jct': AcceptableJCT()}[spec['actor']]
    done, n_env_steps, actions = False, 0, []
    while not done:
        job_to_place = list(env.cluster.job_queue.jobs.values())[0]
        a = actor.compute_action(obs, job_to_place=job_to_place)
        actions.append(int(a))
        obs, _, done, _ = env.step(int(a))
        n_env_steps += 1
    out = cluster_result(env.cluster, n_env_steps, actions, is_dropin=not use_reference_cluster,
                         using_reference_classes=host.USING_REFERENCE_CLASSES)
    if recorder is not None:
        recorder.save(record_path, n_env_steps, actions)
    print('RESULT ' + json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
