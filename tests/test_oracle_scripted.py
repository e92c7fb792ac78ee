"""The CPU oracle's threaded scripted driver (oracle.run_scripted / orc_run_scripted_rjpe_batch_ex), which the GPU tests take
as the reference for whole batches of scripted episodes, against a plain Python loop over one OracleEnv per episode."""
import copy

import numpy as np
import pytest

from workload_script import script_of

CONFIGS = ['cfg1-chain-8w', 'cfg2-resnet50-32w']


def _workload(config, oracle_lib, B=6, L=8, seed=3):
    from ddls_b200 import workload
    jcts = lambda ts: [oracle_lib.run_lookahead(t, trace_cap=0)['jct'] for t in ts]
    # exponential gaps: some jobs arrive while others run, so env-steps take different numbers of cluster steps
    wl = workload.generate(config, jcts, n_episodes=B, n_steps=L, seed=seed, interarrival=400.0)
    rng = np.random.default_rng(seed)
    wl.arrivals['interarrival'][:, :-1] = rng.exponential(400.0, size=(B, L - 1))
    return wl


def _python_rollout(oracle_lib, wl, tid, mount, b):
    """RampJobPartitioningEnvironment.step (RJPE:300-420) spelled out: the action step, then Action() while no job is queued
    and the episode is not done."""
    from ddls_b200.lowered import MountScalars
    L = tid.shape[1]
    n_models = max(wl.template_model) + 1
    env = oracle_lib.OracleEnv(wl.shape.n_workers, max_jobs=wl.arrivals.shape[1], memo_models=n_models)
    env.reset(wl.arrivals[b])
    stats, ncs = np.zeros((L, oracle_lib.STEP_STATS_LEN)), np.zeros(L, dtype=np.int32)
    for s in range(L):
        job = None
        if tid[b, s] >= 0 and env.queued_job >= 0:
            job = copy.copy(wl.templates[tid[b, s]])
            m = mount[b, s]
            job.mount = MountScalars(*(m[f].item() for f in mount.dtype.names))
        st = env.step(job)
        last, n = st, 1
        while env.queued_job < 0 and last[oracle_lib.SS['done']] == 0.0:
            last = env.step(None)
            n += 1
        st[oracle_lib.SS['done']] = last[oracle_lib.SS['done']]
        stats[s], ncs[s] = st, n
    return stats, env.job_records(), ncs


@pytest.mark.parametrize('config', CONFIGS)
def test_run_scripted_equals_python_loop(config, oracle_lib):
    wl = _workload(config, oracle_lib)
    tid, mount = script_of(wl)
    n_models = max(wl.template_model) + 1
    stats, rec, ncs = oracle_lib.run_scripted(wl.templates, tid, mount, wl.arrivals, wl.shape.n_workers, n_models, n_threads=3)
    assert stats.shape == (wl.n_episodes, wl.n_steps, oracle_lib.STEP_STATS_LEN) and ncs.shape == tid.shape
    assert (tid >= 0).any() and (ncs > 1).any(), 'the script should place jobs and have env-steps with Action() steps'
    for b in range(wl.n_episodes):
        st_b, rec_b, ncs_b = _python_rollout(oracle_lib, wl, tid, mount, b)
        np.testing.assert_array_equal(stats[b], st_b, err_msg=f'{config} episode {b}')
        np.testing.assert_array_equal(ncs[b], ncs_b, err_msg=f'{config} episode {b}')
        for f in rec.dtype.names:
            np.testing.assert_array_equal(rec[b][f], rec_b[f], err_msg=f'{config} episode {b} record field {f}')


@pytest.mark.parametrize('config', CONFIGS)
def test_run_scripted_stats_equal_the_entry_point_without_cluster_steps(config, oracle_lib):
    """orc_run_scripted_rjpe_batch (the call the CPU baseline times) and the _ex variant compute the same episodes."""
    wl = _workload(config, oracle_lib, B=16)
    tid, mount = script_of(wl)
    n_models = max(wl.template_model) + 1
    stats, rec, _ = oracle_lib.run_scripted(wl.templates, tid, mount, wl.arrivals, wl.shape.n_workers, n_models, n_threads=4)
    keep = [oracle_lib.to_c(t) for t in wl.templates]
    ctemps = (oracle_lib.CLoweredJob * len(keep))(*keep)
    arr = np.ascontiguousarray(wl.arrivals, dtype=oracle_lib.ARRIVAL_DTYPE)
    old = np.zeros_like(stats)
    old_rec = np.zeros_like(rec)
    rc = oracle_lib.lib().orc_run_scripted_rjpe_batch(ctemps, len(keep), tid.shape[0], tid.shape[1], tid.ctypes.data,
                                                      mount.ctypes.data, arr.ctypes.data, arr.shape[1], float('inf'),
                                                      wl.shape.n_workers, n_models, 1025, old.ctypes.data, old_rec.ctypes.data, 2)
    assert rc == 0
    np.testing.assert_array_equal(stats, old)
    for f in rec.dtype.names:
        np.testing.assert_array_equal(rec[f], old_rec[f])
