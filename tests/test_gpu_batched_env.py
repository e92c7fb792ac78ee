"""-m gpu: ``ddls_b200.batched.BatchedRampJobPartitioningEnvironment`` -- B RampJobPartitioningEnvironment episodes in lock step on
one engine, every decision lowered by the native placer + native expansion (no reference objects) -- replays the reference's
recorded golden episodes SIDE BY SIDE in one batch: same arrival streams, same actions (the partition degrees the reference's
actors chose), and must reproduce what the reference recorded for each episode: the statistics of every env-step's first
cluster step, which jobs completed / were blocked, every job completion time and overhead (<= 1e-6 relative), and every
env-step's reward against the reference's rule evaluated on the CPU oracle replaying the same episode."""
import numpy as np
import pytest

from golden_io import Golden

pytestmark = pytest.mark.gpu


def _graphs():
    from ddls_b200 import synth
    return {
        'chain8': [synth.chain_graph(6, 'chain6')], 'chain8_busy': [synth.chain_graph(6, 'chain6')],
        'chain8_maxtime': [synth.chain_graph(6, 'chain6')], 'residual8_deg4': [synth.residual_small_graph()],
        'mixed16': [synth.chain_graph(5, 'chain5'), synth.resnet_like_graph(n_blocks=2, stem=2, name='res2', seed=7, body_per_block=3),
                    synth.transformer_like_graph(n_layers=1, name='tfm1', seed=4)],
        'tfm32_acceptable': [synth.transformer_like_graph(n_layers=2, name='tfm2', seed=9)],
        'mixed64_busy': [synth.chain_graph(4, 'chain4'), synth.resnet_like_graph(n_blocks=1, stem=2, name='res1', seed=11, body_per_block=2),
                         synth.transformer_like_graph(n_layers=1, name='tfm1b', seed=6)],
        'res16_flood': [synth.resnet_like_graph(n_blocks=1, stem=1, name='res1s', seed=3, body_per_block=2)],
        'residual32_deg16': [synth.residual_small_graph()],
        'resnet64_deg16_full': [synth.resnet_like_graph()], 'resnet64_deg8_full': [synth.resnet_like_graph()],
        'resnet64_deg4_full': [synth.resnet_like_graph()], 'resnet64_deg2_full': [synth.resnet_like_graph()],
        # BASELINE configs 4 / 5: 256- and 128-worker clusters (occupancy bit sets of 4 and 2 words)
        'resnet32_cfg2': [synth.resnet_like_graph()],
        'bert256_shard': [synth.transformer_like_graph(n_layers=12, name='bert_base_like', seed=2)],
        'mix128_exp': [synth.resnet_like_graph(), synth.transformer_like_graph(n_layers=12, name='gpt2_small_like', seed=5, gpt=True)],
    }


SHAPES = {8: (2, 2, 2), 16: (2, 2, 4), 32: (4, 4, 2), 64: (4, 4, 4), 128: (8, 4, 4), 256: (8, 8, 4)}
# episodes that share a topology and a max_simulation_run_time run in ONE batch
BATCHES = [
    ['chain8', 'chain8_busy', 'residual8_deg4', 'chain8', 'chain8_busy'],
    ['chain8_maxtime'],
    ['mixed16', 'res16_flood', 'mixed16'],
    ['tfm32_acceptable', 'residual32_deg16', 'resnet32_cfg2'],
    ['mixed64_busy', 'resnet64_deg2_full', 'resnet64_deg4_full', 'resnet64_deg8_full', 'resnet64_deg16_full'],
    ['mix128_exp', 'mix128_exp'],
    ['bert256_shard'],
]


def _decisions(g):
    """Per env-step: (index of its first cluster step, action = max partition degree or 0)."""
    from ddls_b200.engine import SS
    ref, tids = g.d['step_stats'], g.d['step_tid']
    out, s = [], 0
    while s < g.n_steps:
        tid = int(tids[s])
        out.append((s, g.templates[tid].degree if tid >= 0 else 0))
        s += 1
        while s < g.n_steps and ref[s - 1, SS['job_queue_length']] == 0 and ref[s - 1, SS['done']] == 0:
            s += 1
    return out


@pytest.mark.parametrize('where', ['host', 'device'])
@pytest.mark.parametrize('names', BATCHES, ids=lambda n: '+'.join(n))
def test_batched_env_replays_reference_episodes_in_lock_step(names, where):
    """where='host': placement / lowering / bookkeeping in numpy + native C++ on the host; 'device': the ramp_env_* kernels (first-fit
    over candidate blocks, template table, reward, occupancy, observation features on the GPU)."""
    from ddls_b200 import batched
    BatchedRampJobPartitioningEnvironment = (batched.BatchedRampJobPartitioningEnvironment if where == 'host'
                                             else batched.DeviceRampJobPartitioningEnvironment)
    from ddls_b200.engine import SS, JS_COMPLETED, JS_BLOCKED
    from ddls_b200.template_builder import original_job_totals
    goldens = [Golden(n) for n in names]
    n_workers = goldens[0].n_cluster_workers
    assert all(g.n_cluster_workers == n_workers and g.max_sim_time == goldens[0].max_sim_time for g in goldens)
    catalogue = _graphs()
    graphs, seen = [], {}
    for n in names:
        for gr in catalogue[n]:
            if gr.name not in seen:
                seen[gr.name] = len(graphs)
                graphs.append(gr)
    totals = [original_job_totals(gr)[0] for gr in graphs]
    B = len(goldens)
    J = max(len(g.d['arrivals']) for g in goldens)
    model = np.zeros((B, J), dtype=np.int64)
    gap = np.full((B, J), np.inf)
    macc = np.full((B, J), np.nan)
    decisions = []
    for b, (n, g) in enumerate(zip(names, goldens)):
        arr = g.d['arrivals']
        for k in range(len(arr)):
            cands = [seen[gr.name] for gr in catalogue[n] if abs(totals[seen[gr.name]] - arr[k, 1]) <= 1e-9 * abs(arr[k, 1])]
            assert len(cands) == 1, (n, k)
            model[b, k] = cands[0]
            gap[b, k] = arr[k, 0]
        dec = _decisions(g)
        decisions.append(dec)
        # the job handled by env-step e is job e (one decision per arrival); its max acceptable JCT as the reference computed it
        for e, (s, a) in enumerate(dec):
            if a > 0:
                macc[b, e] = g.d['step_mount'][s][0]
    env = BatchedRampJobPartitioningEnvironment(SHAPES[n_workers], graphs, n_episodes=B, jobs_per_episode=J, max_partitions_per_op=16,
                                                max_simulation_run_time=goldens[0].max_sim_time,
                                                script={'model': model, 'gap': gap, 'max_acceptable_jct': macc}, apply_action_mask=False)
    obs = env.reset()
    for b, g in enumerate(goldens):
        env.eng.set_job_count(b, len(g.d['arrivals']))
    # each golden episode replayed on the CPU oracle beside the batch: it says whether a placed job was blocked by the end of its
    # action's cluster step, which is what the reference's reward looks at (RJPE:379-391, rewards/job_acceptance.py)
    from oracle import oracle
    oracle.build()
    oenvs = []
    for g in goldens:
        oe = oracle.OracleEnv(g.n_cluster_workers, max_jobs=len(g.arrivals()), memo_models=max(g.n_models, 1))
        oe.reset(g.arrivals(), max_simulation_run_time=g.max_sim_time)
        oenvs.append(oe)
    n_env_steps = max(len(d) for d in decisions)
    exact = ['num_jobs_completed', 'num_jobs_arrived', 'num_jobs_blocked']
    close = ['step_start_time', 'step_end_time', 'mean_num_jobs_running', 'mean_compute_overhead_frac', 'mean_communication_overhead_frac',
             'compute_info_processed', 'dep_info_processed', 'flow_info_processed', 'mean_cluster_throughput', 'mean_num_mounted_workers']
    for e in range(n_env_steps):
        actions = np.zeros(B, dtype=np.int64)
        for b in range(B):
            if e < len(decisions[b]):
                assert not env.done[b], (names[b], e)
                assert env.queued[b] == e
                actions[b] = decisions[b][e][1]
            else:
                assert env.done[b], (names[b], e)
        obs, reward, done, info = env.step(actions)
        for b, g in enumerate(goldens):
            if e >= len(decisions[b]):
                assert reward[b] == 0.0, (names[b], e, reward[b])        # the episode was already done
                continue
            s = decisions[b][e][0]
            ref = g.d['step_stats'][s]
            st = env.last_stats[b]
            for k in exact:
                assert st[SS[k]] == ref[SS[k]], (names[b], e, k, st[SS[k]], ref[SS[k]])
            for k in close:
                assert st[SS[k]] == pytest.approx(ref[SS[k]], rel=1e-6, abs=0), (names[b], e, k)
            # the reference's reward: success iff the decision placed the job and the job is not blocked after the action's
            # cluster step, else fail (RJPE:379-391, rewards/job_acceptance.py)
            placed = decisions[b][e][1] > 0 and int(g.d['step_tid'][s]) >= 0
            oe = oenvs[b]
            assert oe.queued_job == e, (names[b], e, oe.queued_job)
            o = oe.step(g.step_job(s) if placed else None)
            blocked = oe.job_records()['status'][e] == JS_BLOCKED
            want = env.success_reward if placed and not blocked else env.fail_reward
            assert reward[b] == want, (where, names[b], e, 'placed' if placed else 'not placed', 'blocked' if blocked else '',
                                       reward[b], want)
            while oe.queued_job < 0 and o[SS['done']] == 0.0:                # RJPE:394-395
                o = oe.step(None)
    assert env.done.all()
    rec = env.eng.job_records()
    for b, g in enumerate(goldens):
        r = rec[b][:len(g.d['arrivals'])]
        order = np.argsort(r['event_seq'], kind='stable')
        completed = [int(i) for i in order if r['status'][i] == JS_COMPLETED]
        blocked = [int(i) for i in order if r['status'][i] == JS_BLOCKED]
        assert completed == list(g.d['es_completed_job_idxs']), names[b]
        assert sorted(blocked) == sorted(g.d['es_blocked_job_idxs']), names[b]
        np.testing.assert_allclose(r['time_completed'][completed] - r['time_arrived'][completed], g.d['es_job_completion_time'], rtol=1e-6, atol=0)
        np.testing.assert_allclose(r['comm'][completed], g.d['es_job_communication_overhead_time'], rtol=1e-6, atol=0)
        np.testing.assert_allclose(r['comp'][completed], g.d['es_job_computation_overhead_time'], rtol=1e-6, atol=0)
        np.testing.assert_allclose(r['util'][completed], g.d['es_jobs_completed_mean_mounted_worker_utilisation_frac'], rtol=1e-6, atol=0)
    # the batch shared placements and templates: far fewer native calls than decisions
    n_decisions = sum(1 for d in decisions for (_, a) in d if a > 0)
    assert env.stats['placer_calls'] <= n_decisions
    env.close()


def test_device_env_equals_host_env_on_random_rollouts():
    """The device-resident environment against the host one, same streams and actions: rewards, done flags, dynamic observation
    features, action masks and every job record must be identical."""
    from ddls_b200 import synth
    from ddls_b200.batched import BatchedRampJobPartitioningEnvironment, DeviceRampJobPartitioningEnvironment
    graphs = [synth.resnet_like_graph(n_blocks=2, stem=2, name='res2', seed=7, body_per_block=3), synth.chain_graph(6, 'chain6'),
              synth.transformer_like_graph(n_layers=1, name='tfm1', seed=4)]
    kw = dict(n_episodes=768, jobs_per_episode=7, seed=11, interarrival=('exponential', 600.0))
    host = BatchedRampJobPartitioningEnvironment((4, 4, 4), graphs, **kw)
    dev = DeviceRampJobPartitioningEnvironment((4, 4, 4), graphs, **kw)
    oh, od = host.reset(), dev.reset()
    rng = np.random.default_rng(5)
    cand = np.array([0, 1, 2, 4, 8, 16])
    for _ in range(7):
        np.testing.assert_array_equal(oh['action_mask'], od['action_mask'])
        np.testing.assert_array_equal(np.where(oh['done'], -1, oh['model']), np.where(od['done'], -1, od['model']))
        live = ~oh['done']
        np.testing.assert_allclose(oh['graph_features_dynamic'][live], od['graph_features_dynamic'][live], rtol=1e-6, atol=0)
        ok = oh['action_mask'][:, cand].astype(bool)
        r = rng.random(ok.shape) * ok
        actions = cand[r.argmax(axis=1)]
        oh, rh, dh, _ = host.step(actions)
        od, rd, dd, _ = dev.step(actions)
        np.testing.assert_array_equal(rh, rd)
        np.testing.assert_array_equal(dh, dd)
        a, b = host.eng.job_records(), dev.eng.job_records()
        for f in a.dtype.names:
            np.testing.assert_array_equal(a[f], b[f], err_msg=f)
    assert dh.all()
    # the tfm1 model mixes split counts at some degrees: those decisions (and the first use of every block geometry) went to the host
    assert 0 < dev.stats['placer_calls'] < 2000
    host.close(); dev.close()


def test_batched_env_rollout_with_random_policy_is_consistent():
    """4,096-episode random rollouts: rewards, done flags and the occupancy the host keeps agree with the engine's own state."""
    from ddls_b200 import synth
    from ddls_b200.batched import BatchedRampJobPartitioningEnvironment
    from ddls_b200.engine import EP, JS_RUNNING
    env = BatchedRampJobPartitioningEnvironment((4, 4, 4), [synth.resnet_like_graph(n_blocks=2, stem=2, name='res2', seed=7, body_per_block=3),
                                                            synth.chain_graph(6, 'chain6')], n_episodes=512, jobs_per_episode=6, seed=3)
    rng = np.random.default_rng(0)
    obs = env.reset()
    total_reward = np.zeros(512)
    for _ in range(6):
        mask = obs['action_mask'].astype(bool)
        cand = np.array([2, 4, 8, 16])
        ok = mask[:, cand]
        pick = np.array([rng.choice(cand[o]) if o.any() else 0 for o in ok])
        obs, reward, done, info = env.step(pick)
        total_reward += reward
        st = env.eng.episode_state()
        rec = env.eng.job_records()
        assert np.array_equal(env.n_running, (rec['status'] == JS_RUNNING).sum(axis=1))
        assert np.array_equal(env.n_running, st[:, EP['num_running']].astype(np.int64))
        # one job per worker (ramp_rules.py:6-39): the server sets of the running jobs of an episode are disjoint
        running = rec['status'] == JS_RUNNING
        pop = np.bitwise_count(np.where(running[:, :, None], env.job_mask, np.uint64(0))).sum(axis=(1, 2))
        assert np.array_equal(pop, np.bitwise_count(env.busy).sum(axis=1))
    assert done.all()
    assert env.stats['placer_calls'] < 200 and env.stats['expansions'] < 100
    env.close()
