"""-m gpu: the batched step path (ramp_step_device: plan -> bucket -> thread / warp / CTA lookaheads -> step) at benchmark scale,
thousands of different episodes per launch, against the CPU oracle running the same scripted episodes.

  A. the benchmark's own workloads (ddls_b200/workload.py, all five configs at their batch sizes), driven as bench.py drives
     them: two segments with a reset before each, so the second starts with every template's hints recorded;
  B. edges the benchmark does not reach: template ids past 1024, per-template chunk counts around 32, memo hits from jobs
     mounted on a different number of workers, a memo table at ~90 % load and one that overflows;
  C. what bench.py --dump-outputs writes.

Every step-stats column, every job-record field and every cluster-step count must be identical (f64 bit for bit).  Rows of
an episode that is already done follow the engine's skip-row convention instead (the oracle keeps stepping a done env)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from workload_script import engine_actions, script_of

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = 8
BATCH = {'cfg1-chain-8w': 1, 'cfg2-resnet50-32w': 256, 'cfg3-resnet50-64w': 4096, 'cfg4-bert-256w': 4096, 'cfg5-mix-128w': 16384}
MEMO_MODES = {'reference': 0, 'exact': 1, 'off': 2, 'shared': 3}
KNOBS = {'resident0': {'RAMP_RESIDENT': '0'}, 'warp': {'RAMP_LOOKAHEAD_MODE': 'warp'}, 'cta': {'RAMP_LOOKAHEAD_MODE': 'cta'},
         'dense0': {'RAMP_DENSE_FACTOR': '0'}}


def _threads():
    return max(1, len(os.sched_getaffinity(0)))


class Reference:
    """A scripted batch and what the oracle computed for it."""

    def __init__(self, templates, tid, mount, arrivals, n_workers, n_models):
        from oracle import oracle
        oracle.build()
        self.templates, self.tid, self.mount, self.arrivals = templates, tid, mount, arrivals
        self.n_workers, self.n_models = n_workers, n_models
        self.stats, self.rec, self.ncs = oracle.run_scripted(templates, tid, mount, arrivals, n_workers, n_models, _threads())
        self.B, self.L = tid.shape
        # done before env-step s: the oracle's `done` after env-step s - 1
        self.done_before = np.zeros((self.B, self.L), dtype=bool)
        self.done_before[:, 1:] = self.stats[:, :-1, oracle.SS['done']] != 0.0
        self._la = {}

    def lookahead(self, t):
        if t not in self._la:
            from oracle import oracle
            self._la[t] = oracle.run_lookahead(self.templates[t])
        return self._la[t]


def _first_bad(a, b):
    bad = np.argwhere(~((a == b) | (np.isnan(a) & np.isnan(b))))
    return None if len(bad) == 0 else tuple(int(x) for x in bad[0])


def _compare_step(label, ref, s, stats, ncs, memo_mode):
    """stats [B, STEP_STATS_LEN] and ncs [B] of env-step s against the oracle."""
    from ddls_b200.engine import SS, STEP_STATS
    live = ~ref.done_before[:, s]
    cols = [k for k in range(len(STEP_STATS)) if memo_mode == 0 or k != SS['lookahead_ran']]
    got, want = stats[live][:, cols], ref.stats[live, s][:, cols]
    bad = _first_bad(got, want)
    if bad is not None:
        b = int(np.nonzero(live)[0][bad[0]])
        col = STEP_STATS[cols[bad[1]]]
        pytest.fail(f'{label} step {s} episode {b} column {col}: engine {got[bad]!r} oracle {want[bad]!r}')
    bad = np.nonzero(ncs[live] != ref.ncs[live, s])[0]
    if len(bad):
        b = int(np.nonzero(live)[0][bad[0]])
        pytest.fail(f'{label} step {s} episode {b} cluster steps: engine {ncs[b]} oracle {ref.ncs[b, s]}')
    # skip rows (ramp_step_kernel): only done, the step counter and the queue length are written, no cluster step is taken
    done = ref.done_before[:, s]
    if done.any():
        want_row = np.zeros((int(done.sum()), len(STEP_STATS)))
        want_row[:, SS['done']] = 1.0
        ref_ncs = np.where(ref.done_before[:, :s], 0, ref.ncs[:, :s]).sum(axis=1)   # every cluster step the episode took
        want_row[:, SS['step_counter']] = ref_ncs[done]
        bad = _first_bad(stats[done], want_row)
        if bad is not None:
            b = int(np.nonzero(done)[0][bad[0]])
            pytest.fail(f'{label} step {s} episode {b} (done) column {STEP_STATS[bad[1]]}: engine {stats[done][bad]!r} '
                        f'skip row {want_row[bad]!r}')
        assert (ncs[done] == 0).all(), f'{label} step {s}: a done episode took a cluster step'


def _compare_records(label, ref, rec):
    for f in ref.rec.dtype.names:
        bad = _first_bad(rec[f][:, :ref.rec.shape[1]], ref.rec[f])
        if bad is not None:
            pytest.fail(f'{label} job record episode {bad[0]} job {bad[1]} field {f}: engine {rec[f][bad]!r} oracle {ref.rec[f][bad]!r}')


def _compare_lookaheads(label, eng, ref, s, stats, rng, n=256):
    """eng.last_lookahead(b) of a sample of the episodes whose env-step s ran a lookahead (reference memo mode)."""
    from ddls_b200.engine import SS
    ran = np.nonzero((stats[:, SS['lookahead_ran']] == 1.0) & ~ref.done_before[:, s])[0]
    for b in rng.permutation(ran)[:n]:
        la = eng.last_lookahead(int(b))
        o = ref.lookahead(int(ref.tid[b, s]))
        what = f'{label} step {s} episode {b} template {ref.tid[b, s]}'
        assert la['status'] == o['status'] == 0, what
        assert (la['jct'], la['comm'], la['comp'], la['n_ticks']) == (o['jct'], o['comm'], o['comp'], o['n_ticks']), what
        np.testing.assert_array_equal(la['trace_n_active'], o['trace_n_active'][:eng.trace_cap], err_msg=what)
        np.testing.assert_array_equal(la['trace_tick'], o['trace_tick'][:eng.trace_cap], err_msg=what)


def _make_engine(ref, memo_mode, env=None, **kw):
    from ddls_b200 import engine
    for k, v in (env or {}).items():
        os.environ[k] = v
    try:
        eng = engine.RampEngine(n_episodes=ref.B, n_cluster_workers=ref.n_workers, max_jobs=ref.arrivals.shape[1],
                                memo_mode=memo_mode, trace_cap=4096, **kw)
    finally:
        for k in (env or {}):
            os.environ.pop(k, None)
    tmap = [eng.register_template(t) for t in ref.templates]
    return eng, tmap


def _run(label, ref, memo_mode, entry, env=None, segments=2, check_lookaheads=False, **kw):
    """Drives the scripted batch through one engine, `segments` times with a reset before each (bench.py:run_b200_arm)."""
    import torch
    from ddls_b200 import engine
    eng, tmap = _make_engine(ref, memo_mode, env, **kw)
    try:
        actions = engine_actions(engine, ref.tid, ref.mount, tmap)
        B = ref.B
        if entry == 'step_device':
            on_dev = [torch.from_numpy(a.view(np.uint8).reshape(B, -1).copy()).cuda() for a in actions]
            stats_dev = torch.empty((B, engine.STEP_STATS_LEN), dtype=torch.float64, device='cuda')
            ncs_dev = torch.empty(B, dtype=torch.int32, device='cuda')
            torch.cuda.synchronize()
        rng = np.random.default_rng(0)
        for seg in range(segments):
            eng.reset(ref.arrivals)
            for s in range(ref.L):
                if entry == 'step_device':
                    eng.step_device(on_dev[s].data_ptr(), True, stats_dev.data_ptr(), ncs_dev.data_ptr())
                    eng.sync()
                    stats, ncs = stats_dev.cpu().numpy(), ncs_dev.cpu().numpy()
                else:
                    stats, ncs = eng.step(actions[s], fuse_empty_steps=True, want_cluster_steps=True)
                eng.check_status()
                _compare_step(f'{label} segment {seg}', ref, s, stats, ncs, memo_mode)
                if check_lookaheads:
                    _compare_lookaheads(f'{label} segment {seg}', eng, ref, s, stats, rng)
            _compare_records(f'{label} segment {seg}', ref, eng.job_records())
        return eng.memo_stats_ex()
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# A. the benchmark's workloads

_REFS = {}


def _bench_reference(config):
    if config not in _REFS:
        from ddls_b200 import workload
        from oracle import oracle
        oracle.build()
        jcts = lambda ts: [oracle.run_lookahead(t, trace_cap=0)['jct'] for t in ts]
        wl = workload.generate(config, jcts, n_episodes=BATCH[config], n_steps=L, seed=0, run_times='reference')
        tid, mount = script_of(wl)
        _REFS[config] = Reference(wl.templates, tid, mount, wl.arrivals, wl.shape.n_workers, max(wl.template_model) + 1)
    return _REFS[config]


# the bench's `value` (device-resident action rows) and `e2e_engine` (host buffers) entry points
CASES = [(c, m, 'default', e) for c in BATCH for m in MEMO_MODES for e in ('step_device', 'step')] + \
        [(c, 'reference', k, e) for c in ('cfg3-resnet50-64w', 'cfg4-bert-256w') for k in KNOBS for e in ('step_device', 'step')]


@pytest.mark.parametrize('config,memo,knob,entry', CASES, ids=['-'.join(c) for c in CASES])
def test_benchmark_workload_vs_oracle(config, memo, knob, entry):
    """These workloads lower one job per (model, degree), so every memo mode must give the reference's numbers."""
    ref = _bench_reference(config)
    assert (ref.tid >= 0).any()
    check = memo == 'reference' and knob == 'default' and entry == 'step_device'
    _run(f'{config} memo={memo} knob={knob} entry={entry}', ref, MEMO_MODES[memo], entry, env=KNOBS.get(knob),
         check_lookaheads=check)


# ---------------------------------------------------------------------------------------------------------------------
# B. edges the benchmark does not reach

EDGE_B = 4096
EDGE_COUNTS = [1, 31, 32, 33, 64, 65]


@pytest.fixture(scope='module')
def edge_reference():
    """B = 4,096 episodes of 8 jobs on a 256-worker RAMP over ~1,100 registered templates: a decision for each job, then
    one more for the episode that is done by then.

    Templates: cheap random lowered jobs (general path, no symmetry) whose (model, degree) keys are shared by about two
    jobs each, six symmetric ResNet- and chain-like jobs (resident symmetry quotient) and the BERT-like degree-16 job of
    config 4 (not resident), the last seven with ids past 1024.  Each episode picks 7 or 8 distinct keys over its 8
    decisions: a repeated key is a memo hit, usually from a different job and usually mounted on a different number of
    workers (drawn per decision), so its utilisation is recomputed from the pooled trace.  The reference-mode memo holds
    sum(distinct keys) ~ 0.9 x 2^15 entries at the end of the segment.  Env-step 0 gives the symmetric jobs 1, 31, 32, 33,
    64 and 65 lookaheads (partial and exact chunks of 32) beside non-resident work."""
    from ddls_b200 import synth, workload
    from ddls_b200.template_builder import RampShape, build_template, random_dag_template
    from oracle import oracle
    oracle.build()
    rng = np.random.default_rng(2024)
    n_keys_m, n_keys_d = 24, 24
    rand = []
    k = 0
    while len(rand) < 1100:
        t = random_dag_template(rng, int(rng.integers(2, 40)), n_workers=int(rng.integers(1, 5)),
                               model_id=k % n_keys_m, degree=(k // n_keys_m) % n_keys_d)
        k += 1
        if oracle.run_lookahead(t)['status'] == 0:
            rand.append(t)
    shape = RampShape(8, 8, 4)
    g = synth.resnet_like_graph(n_blocks=2, stem=2, name='res2', seed=7, body_per_block=3)
    sym = [build_template(g, d, RampShape(4, 4, 4), model_id=n_keys_m) for d in (2, 4, 8, 16)]
    sym += [build_template(synth.chain_graph(6, 'chain6'), d, RampShape(4, 4, 4), model_id=n_keys_m + 1) for d in (2, 4)]
    bert = workload.build_templates('cfg4-bert-256w', run_times='reference')[3][-1]
    assert bert.degree == 16
    bert.model_id = n_keys_m + 2
    templates = rand + sym + [bert]
    n_rand = len(rand)
    big = list(range(n_rand, len(templates)))
    assert big[0] >= 1024
    keys = np.array([(t.model_id, t.degree) for t in templates])
    key_id = keys[:, 0] * 1025 + keys[:, 1]
    by_key = {}
    for i in range(n_rand):
        by_key.setdefault(int(key_id[i]), []).append(i)
    key_list = list(by_key)

    B = EDGE_B
    tid = np.zeros((B, L + 1), dtype=np.int32)
    for b in range(B):
        n_distinct = 8 if rng.random() < 0.2 else 7
        ks = rng.choice(len(key_list), size=n_distinct, replace=False)
        picks = [int(rng.choice(by_key[key_list[j]])) for j in ks]
        if n_distinct == 7:                                  # a second job of one of the keys already used, later
            j = int(rng.integers(0, 6))
            picks.insert(int(rng.integers(j + 1, 8)), int(rng.choice(by_key[key_list[ks[j]]])))
        tid[b, :L] = picks
    tid[:, L] = rng.integers(-1, len(templates), size=B)      # a decision after the episode is done: a skip row
    # env-step 0: the symmetric jobs with the chunk-boundary counts, the non-resident job beside them
    e = 0
    counts = dict(zip(big[:6], EDGE_COUNTS))
    for t, c in counts.items():
        tid[e:e + c, 0] = t
        e += c
    tid[e:e + 24, 0] = big[6]
    e += 24
    tid[rng.permutation(B)[:24], 5] = big[6]                  # the non-resident job again later, as a memo miss
    assert e < B
    # mount scalars: a mounted-worker count drawn per decision, max acceptable JCT a random fraction of the job's own lookahead
    jct = np.array([oracle.run_lookahead(t, trace_cap=0)['jct'] for t in templates])
    from oracle.oracle import MOUNT_DTYPE
    mount = np.zeros(tid.shape, dtype=MOUNT_DTYPE)
    mount['max_acceptable_jct'] = np.round(rng.uniform(0.3, 1.7, size=tid.shape), 2) * jct[tid]
    mount['part_op_mem'] = rng.uniform(1.0, 100.0, size=tid.shape)
    mount['part_dep_size'] = rng.uniform(1.0, 100.0, size=tid.shape)
    mount['flow_size'] = mount['part_dep_size'] * 0.5
    mount['n_mounted_workers'] = rng.integers(1, 17, size=tid.shape)
    mount['n_mounted_channels'] = rng.integers(0, 9, size=tid.shape)
    arrivals = np.zeros((B, L), dtype=oracle.ARRIVAL_DTYPE)
    arrivals['interarrival'] = rng.exponential(np.median(jct) * 0.5, size=(B, L))
    arrivals['interarrival'][:, -1] = np.inf
    arrivals['orig_op_mem'] = rng.uniform(50.0, 500.0, size=(B, L))
    arrivals['orig_dep_size'] = rng.uniform(50.0, 500.0, size=(B, L))
    return Reference(templates, tid, mount, arrivals, shape.n_workers, n_keys_m + 3)


def test_edge_workload_is_what_it_claims(edge_reference):
    from oracle.oracle import SS, JS_BLOCKED, JS_COMPLETED
    ref = edge_reference
    assert not ref.done_before[:, :L].any(), 'every env-step but the last should handle a queued job'
    assert ref.done_before[:, L].all()
    ran = ref.stats[:, :, SS['lookahead_ran']]
    assert ran.sum() / 2 ** 15 == pytest.approx(0.9, abs=0.02)
    assert (ran[:, 0] == 1).all() and (ran == 0).any()                           # memo hits
    blocked = (ref.rec['status'] == JS_BLOCKED).sum()
    assert 0.1 * ref.rec.size < blocked < 0.9 * ref.rec.size
    assert (ref.rec['status'] == JS_COMPLETED).any()
    assert (ref.ncs > 1).any()


@pytest.mark.parametrize('memo', ['reference', 'shared'])
def test_edge_workload_vs_oracle(memo, edge_reference):
    """max_templates = 2048 (ids past 1024: the bucket kernel's multi-round scan), memo table at ~90 % load (long probes)."""
    m = _run(f'edge memo={memo}', edge_reference, MEMO_MODES[memo], 'step_device', max_templates=2048, memo_capacity_log2=15,
             check_lookaheads=(memo == 'reference'))
    if memo == 'reference':
        assert m['lookaheads'] == int(edge_reference.stats[:, :, -1].sum())


def test_memo_table_overflow_is_reported(edge_reference):
    """A table that cannot hold every (episode, model, degree) key: the plan kernel reports TABLE_FULL through check_status."""
    from ddls_b200 import engine
    ref = edge_reference
    eng, tmap = _make_engine(ref, MEMO_MODES['reference'], max_templates=2048, memo_capacity_log2=11)
    try:
        a = engine_actions(engine, ref.tid, ref.mount, tmap)[0]
        eng.reset(ref.arrivals)
        eng.step(a, fuse_empty_steps=True)
        with pytest.raises(Exception, match='memo table is full'):
            eng.check_status()
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# C. bench.py --dump-outputs

def test_bench_dump_outputs_vs_oracle(tmp_path):
    W, K, B, config = 3, 10, 512, 'cfg3-resnet50-64w'
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--episodes', str(B), '--warmup', str(W), '--steps', str(K),
           '--no-cpu-baseline', '--no-batched-env', '--dump-outputs', str(tmp_path)]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stderr[-3000:]
    stats = np.load(tmp_path / 'step_stats.npy')
    ncs = np.load(tmp_path / 'cluster_steps.npy')
    from ddls_b200 import workload
    from oracle import oracle
    oracle.build()
    jcts = lambda ts: [oracle.run_lookahead(t, trace_cap=0)['jct'] for t in ts]
    wl = workload.generate(config, jcts, n_episodes=B, n_steps=L, seed=0, run_times='reference')
    tid, mount = script_of(wl)
    ref = Reference(wl.templates, tid, mount, wl.arrivals, wl.shape.n_workers, max(wl.template_model) + 1)
    s = (W + K - 1) % L
    assert stats.shape == (B, oracle.STEP_STATS_LEN) and ncs.shape == (B,)
    _compare_step(f'bench.py --dump-outputs ({config}, B={B}, env-step {s})', ref, s, stats, ncs.astype(np.int32), memo_mode=0)
