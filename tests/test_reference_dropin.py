"""The drop-in ``ddls_b200.host.RampClusterEnvironment`` driven the way the UNMODIFIED reference drives it: its
RampJobPartitioningEnvironment (RJPE:199-206 swapped to the drop-in), first-fit placers, SRPT schedulers, Job and
JobsGenerator classes, on the seeded golden episodes.  Everything the reference handed to the drop-in in those episodes is
stored as a session (tests/golden/dropin/<case>.npz, recorded by tests/ref_dropin_driver.py --record) and replayed by
tests/dropin_replay.py; the per-step log and the episode statistics must equal what the reference recorded for itself
(tests/golden/<case>.npz, written by oracle/gen_golden.py), or what the reference's own cluster environment produced on the
same episode (tests/golden/dropin/<case>_reference.json, tests/ref_dropin_driver.py --reference-cluster).

The CPU variant answers the engine calls with the oracle (tests/fake_engine.py): it checks the HOST logic (mount
bookkeeping, lowering of reference-shaped Action objects, arrival streaming, replay into episode_stats, the init-details
memo).  The ``-m gpu`` variant is the same run on the CUDA engine."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from golden_io import Golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ['chain8', 'chain8_busy', 'chain8_maxtime', 'mixed16', 'res16_flood', 'residual8_deg4', 'tfm32_acceptable', 'mixed64_busy',
         'mix128_exp',            # 128 workers, exponential arrivals (BASELINE config 5 in small)
         'resnet32_cfg2']         # BASELINE config 2's cluster and job (32 workers, ResNet-50-like), degrees 4 / 6 / 8


def _run(case, fake):
    """The drop-in's result on the recorded session of ``case``."""
    cmd = [sys.executable, os.path.join(ROOT, 'tests', 'dropin_replay.py'), case] + (['--fake-engine'] if fake else [])
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, env=dict(os.environ, PYTHONHASHSEED='0'))
    lines = [l for l in p.stdout.splitlines() if l.startswith('RESULT ')]
    assert p.returncode == 0 and lines, (p.stdout[-2000:], p.stderr[-4000:])
    return json.loads(lines[-1][len('RESULT '):])


def _reference_result(case):
    """The reference's own cluster environment on the same episode (recorded live)."""
    with open(os.path.join(ROOT, 'tests', 'golden', 'dropin', f'{case}_reference.json')) as f:
        return json.load(f)


def _check(case, out):
    g = Golden(case)
    d = g.d
    assert out['num_jobs_arrived'] == int(d['es_num_jobs_arrived'])
    assert out['num_jobs_completed'] == int(d['es_num_jobs_completed'])
    assert out['num_jobs_blocked'] == int(d['es_num_jobs_blocked'])
    assert out['n_env_steps'] == int(d['meta_n_env_steps'])
    assert out['completed_job_idxs'] == [int(x) for x in d['es_completed_job_idxs']]
    assert sorted(out['blocked_job_idxs']) == sorted(int(x) for x in d['es_blocked_job_idxs'])
    for k in ('episode_end_time', 'mean_load_rate', 'blocking_rate', 'acceptance_rate', 'compute_info_processed', 'dep_info_processed',
              'flow_info_processed', 'cluster_info_processed', 'mean_compute_throughput', 'mean_cluster_throughput',
              'mean_compute_overhead_frac', 'mean_communication_overhead_frac', 'mean_num_jobs_running', 'mean_num_mounted_workers'):
        assert out[k] == pytest.approx(float(d[f'es_{k}']), rel=1e-6, abs=0), k
    for k in ('job_completion_time', 'job_completion_time_speedup', 'job_communication_overhead_time', 'job_computation_overhead_time',
              'jobs_completed_mean_mounted_worker_utilisation_frac', 'jobs_completed_num_mounted_workers',
              'jobs_completed_num_mounted_channels', 'jobs_completed_max_acceptable_job_completion_time',
              'jobs_blocked_max_acceptable_job_completion_time'):
        np.testing.assert_allclose(out[k], d[f'es_{k}'], rtol=1e-6, atol=0, err_msg=k)
    # per cluster step (RCE:1082-1109 steps_log) against the recorded step_stats rows
    from oracle.oracle import SS
    ref = d['step_stats']
    log = out['steps_log']
    assert len(log['step_end_time']) == len(ref)
    for k in log:
        a, b = np.array(log[k]), ref[:, SS[k]]
        if k == 'num_jobs_blocked':       # the log is appended before the jobs still running at the end of the simulation are
            a, b = a[:-1], b[:-1]         # blocked (RCE:1082-1090 vs RCE:1111-1121); the recorded rows are the final step_stats
        np.testing.assert_allclose(a, b, rtol=1e-6, atol=0, err_msg=k)
    for k, v in out['last_step_stats'].items():
        assert v == pytest.approx(float(ref[-1, SS[k]]), rel=1e-6, abs=0), k
    # the two per-tick lists (RCE:989-994): the goldens hold each step's sum and length
    for k, k_sum in (('mean_mounted_worker_utilisation_frac', 'util_mounted_sum'), ('mean_cluster_worker_utilisation_frac', 'util_cluster_sum')):
        lists = out['tick_lists'][k]
        assert [len(x) for x in lists] == [int(n) for n in ref[:, SS['num_ticks']]]
        np.testing.assert_allclose([float(np.sum(x)) for x in lists], ref[:, SS[k_sum]], rtol=1e-9, atol=1e-12, err_msg=k)
    # RCE:876-879: one init-details entry per (model, max partition degree) whose lookahead was accepted
    assert len(out['init_details_memo_keys']) >= 1 or out['num_jobs_completed'] == 0


@pytest.mark.parametrize('case', CASES)
def test_dropin_inside_the_reference_host_logic(case):
    out = _run(case, fake=True)
    _check(case, out)


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES)
def test_dropin_inside_the_reference_on_cuda(case):
    out = _run(case, fake=False)
    _check(case, out)


def _check_live(mine, ref):
    """Drop-in vs the reference's own cluster environment run live on the same seeds."""
    assert mine['is_dropin'] and not ref['is_dropin']
    for k in ('num_jobs_arrived', 'num_jobs_completed', 'num_jobs_blocked', 'n_env_steps', 'n_cluster_steps', 'actions',
              'completed_job_idxs'):
        assert mine[k] == ref[k], k
    assert sorted(mine['blocked_job_idxs']) == sorted(ref['blocked_job_idxs'])
    for k in ('episode_end_time', 'mean_load_rate', 'blocking_rate', 'acceptance_rate', 'cluster_info_processed',
              'mean_cluster_throughput', 'mean_num_jobs_running'):
        assert mine[k] == pytest.approx(ref[k], rel=1e-6, abs=0), k
    for k in ('job_completion_time', 'job_communication_overhead_time', 'jobs_completed_mean_mounted_worker_utilisation_frac'):
        np.testing.assert_allclose(mine[k], ref[k], rtol=1e-6, atol=0, err_msg=k)
    for k in mine['steps_log']:
        np.testing.assert_allclose(mine['steps_log'][k], ref['steps_log'][k], rtol=1e-6, atol=0, err_msg=k)
    assert mine['last_step_stats'] == pytest.approx(ref['last_step_stats'], rel=1e-6, abs=0)
    for k in mine['tick_lists']:                                   # entry by entry, not just sum and length
        assert len(mine['tick_lists'][k]) == len(ref['tick_lists'][k])
        for a, b in zip(mine['tick_lists'][k], ref['tick_lists'][k]):
            np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-12, err_msg=k)


@pytest.mark.parametrize('case', ['chain8_busy', 'mixed16'])
def test_per_tick_utilisation_lists_equal_the_reference(case):
    """step_stats['mean_mounted_worker_utilisation_frac'] / ['mean_cluster_worker_utilisation_frac'] stay per-tick lists in the
    reference (RCE:989-994); the drop-in returns the engine's own per-iteration entries (every event ends the reference's step --
    RCE:1003-1044 -- so a list has one entry unless rounding keeps an event from firing; the engine records however many there are)."""
    ref = _reference_result(case)
    mine = _run(case, fake=True)
    assert all(len(step) >= 1 for step in ref['tick_lists']['mean_mounted_worker_utilisation_frac'])
    _check_live(mine, ref)


@pytest.mark.parametrize('case', ['chain8_repeat', 'res16_repeat'])
def test_dropin_with_a_generator_that_never_runs_dry(case):
    """'remove_and_repeat' sampling: len(jobs_generator) never reaches 0, the episode ends on max_simulation_run_time and jobs
    keep arriving until then -- the drop-in streams arrivals one ahead instead of fixing their number at reset."""
    ref = _reference_result(case)
    mine = _run(case, fake=True)
    assert ref['num_jobs_arrived'] > 6            # more arrivals than the 3 / 2 distinct jobs the generator holds
    _check_live(mine, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['chain8_repeat'])
def test_dropin_with_a_generator_that_never_runs_dry_on_cuda(case):
    ref = _reference_result(case)
    mine = _run(case, fake=False)
    _check_live(mine, ref)
