/*
 * TEST INFRASTRUCTURE -- multi-threaded driver around the CPU oracle, used as the
 * reported CPU baseline (bench.py cpu_baseline / --impl reference).  Episodes are
 * independent, so they are spread over host threads with OpenMP.
 */
#include "ramp_oracle.h"
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <stdatomic.h>

/* minimal dynamic-scheduling parallel-for over pthreads (this image's gcc has no libgomp) */
typedef void (*orc_body_fn)(int32_t k, void* ctx);
typedef struct { atomic_int next; int32_t n; orc_body_fn body; void* ctx; } orc_pf_t;
static void* orc_pf_worker(void* arg) {
    orc_pf_t* pf = (orc_pf_t*)arg;
    for (;;) {
        int32_t k = atomic_fetch_add(&pf->next, 1);
        if (k >= pf->n) break;
        pf->body(k, pf->ctx);
    }
    return NULL;
}
static void orc_parallel_for(int32_t n, int32_t n_threads, orc_body_fn body, void* ctx) {
    orc_pf_t pf; atomic_init(&pf.next, 0); pf.n = n; pf.body = body; pf.ctx = ctx;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > n) n_threads = n > 0 ? n : 1;
    if (n_threads > 256) n_threads = 256;
    pthread_t th[256];
    for (int32_t t = 1; t < n_threads; ++t) pthread_create(&th[t], NULL, orc_pf_worker, &pf);
    orc_pf_worker(&pf);
    for (int32_t t = 1; t < n_threads; ++t) pthread_join(th[t], NULL);
}

/* Runs n independent lookaheads (RCE:379-467).  jobs[k] may repeat the same template. */
typedef struct { const orc_lowered_job_t* const* jobs; orc_lookahead_result_t* results; atomic_int bad; } orc_lb_t;
static void orc_lb_body(int32_t k, void* c) {
    orc_lb_t* x = (orc_lb_t*)c;
    if (orc_run_lookahead(x->jobs[k], NULL, NULL, 0, &x->results[k]) != ORC_OK) atomic_store(&x->bad, 1);
}
int orc_run_lookahead_batch(const orc_lowered_job_t* const* jobs, int32_t n,
                            orc_lookahead_result_t* results, int32_t n_threads) {
    orc_lb_t x; x.jobs = jobs; x.results = results; atomic_init(&x.bad, 0);
    orc_parallel_for(n, n_threads, orc_lb_body, &x);
    return atomic_load(&x.bad) ? ORC_ERR_BAD_ARG : ORC_OK;
}

/* Scripted batched episodes: episode b performs n_steps RampClusterEnvironment.step calls;
 * step s of episode b uses template script_tid[b*n_steps+s] (or -1 = Action()) with mount
 * scalars script_mount[b*n_steps+s].  stats_out: [n_episodes][n_steps][ORC_STEP_STATS_LEN]
 * (may be NULL).  Each episode has its own env (own memo), like independent reference envs. */
typedef struct {
    const orc_lowered_job_t* templates; int32_t n_templates, n_steps, n_jobs, n_cluster_workers, memo_models, memo_degrees;
    const int32_t* script_tid; const orc_mount_t* script_mount; const orc_arrival_t* arrivals;
    double max_sim_time; double* stats_out; orc_job_record_t* records_out; int32_t* ncs_out; atomic_int bad; int rjpe;
} orc_sb_t;
static void orc_sb_body(int32_t b, void* c) {
    orc_sb_t* x = (orc_sb_t*)c;
    orc_env_t* env = orc_env_create(x->n_cluster_workers, x->n_cluster_workers > 0 ? x->n_cluster_workers : 1, x->n_jobs,
                                    x->memo_models, x->memo_degrees, 0, 1e-7);
    double local[ORC_STEP_STATS_LEN];
    int bad = 0;
    if (orc_env_reset(env, x->max_sim_time, 10, x->arrivals + (size_t)b * (size_t)x->n_jobs, x->n_jobs) != ORC_OK) bad = 1;
    double scratch[ORC_STEP_STATS_LEN];
    for (int32_t s = 0; s < x->n_steps && !bad; ++s) {
        size_t idx = (size_t)b * (size_t)x->n_steps + (size_t)s;
        int32_t tid = x->script_tid[idx];
        double* st = x->stats_out ? x->stats_out + idx * ORC_STEP_STATS_LEN : local;
        int rc;
        if (tid >= 0 && tid < x->n_templates && orc_env_queued_job(env) >= 0)
            rc = orc_env_step(env, &x->templates[tid], &x->script_mount[idx], st);
        else
            rc = orc_env_step(env, NULL, NULL, st);
        if (rc != ORC_OK) bad = 1;
        int32_t n_cluster_steps = 1;
        if (x->rjpe) {   /* RJPE:394-395: while len(job_queue) == 0 and not done: step(Action()) */
            const double* last = st;
            while (!bad && orc_env_queued_job(env) < 0 && last[SS_DONE] == 0.0) {
                if (orc_env_step(env, NULL, NULL, scratch) != ORC_OK) bad = 1;
                last = scratch;
                ++n_cluster_steps;
            }
            st[SS_DONE] = last[SS_DONE];
        }
        if (x->ncs_out) x->ncs_out[idx] = n_cluster_steps;
    }
    if (x->records_out)
        memcpy(x->records_out + (size_t)b * (size_t)x->n_jobs, orc_env_job_records(env), sizeof(orc_job_record_t) * (size_t)x->n_jobs);
    orc_env_destroy(env);
    if (bad) atomic_store(&x->bad, 1);
}
int orc_run_scripted_batch(const orc_lowered_job_t* templates, int32_t n_templates,
                           int32_t n_episodes, int32_t n_steps,
                           const int32_t* script_tid, const orc_mount_t* script_mount,
                           const orc_arrival_t* arrivals /* [n_episodes][n_jobs] */, int32_t n_jobs,
                           double max_sim_time, int32_t n_cluster_workers, int32_t memo_models, int32_t memo_degrees,
                           double* stats_out, orc_job_record_t* records_out /* [n_episodes][n_jobs] or NULL */,
                           int32_t n_threads) {
    orc_sb_t x;
    x.templates = templates; x.n_templates = n_templates; x.n_steps = n_steps; x.n_jobs = n_jobs;
    x.n_cluster_workers = n_cluster_workers; x.memo_models = memo_models; x.memo_degrees = memo_degrees;
    x.script_tid = script_tid; x.script_mount = script_mount; x.arrivals = arrivals; x.max_sim_time = max_sim_time;
    x.stats_out = stats_out; x.records_out = records_out; x.ncs_out = NULL; atomic_init(&x.bad, 0); x.rjpe = 0;
    orc_parallel_for(n_episodes, n_threads, orc_sb_body, &x);
    return atomic_load(&x.bad) ? ORC_ERR_BAD_ARG : ORC_OK;
}

/* Same, but each scripted decision is one RampJobPartitioningEnvironment.step (RJPE:300-420): the action step
 * followed by Action() steps until a job is queued or the episode is done.  stats_out rows describe the action
 * step (with SS_DONE = done after the whole env-step).  ncs_out [n_episodes][n_steps] (may be NULL): the number of
 * RampClusterEnvironment.step calls each env-step made, the action step included. */
int orc_run_scripted_rjpe_batch_ex(const orc_lowered_job_t* templates, int32_t n_templates,
                                   int32_t n_episodes, int32_t n_steps,
                                   const int32_t* script_tid, const orc_mount_t* script_mount,
                                   const orc_arrival_t* arrivals, int32_t n_jobs,
                                   double max_sim_time, int32_t n_cluster_workers, int32_t memo_models, int32_t memo_degrees,
                                   double* stats_out, orc_job_record_t* records_out, int32_t* ncs_out, int32_t n_threads) {
    orc_sb_t x;
    x.templates = templates; x.n_templates = n_templates; x.n_steps = n_steps; x.n_jobs = n_jobs;
    x.n_cluster_workers = n_cluster_workers; x.memo_models = memo_models; x.memo_degrees = memo_degrees;
    x.script_tid = script_tid; x.script_mount = script_mount; x.arrivals = arrivals; x.max_sim_time = max_sim_time;
    x.stats_out = stats_out; x.records_out = records_out; x.ncs_out = ncs_out; atomic_init(&x.bad, 0); x.rjpe = 1;
    orc_parallel_for(n_episodes, n_threads, orc_sb_body, &x);
    return atomic_load(&x.bad) ? ORC_ERR_BAD_ARG : ORC_OK;
}

int orc_run_scripted_rjpe_batch(const orc_lowered_job_t* templates, int32_t n_templates,
                                int32_t n_episodes, int32_t n_steps,
                                const int32_t* script_tid, const orc_mount_t* script_mount,
                                const orc_arrival_t* arrivals, int32_t n_jobs,
                                double max_sim_time, int32_t n_cluster_workers, int32_t memo_models, int32_t memo_degrees,
                                double* stats_out, orc_job_record_t* records_out, int32_t n_threads) {
    return orc_run_scripted_rjpe_batch_ex(templates, n_templates, n_episodes, n_steps, script_tid, script_mount, arrivals, n_jobs,
                                          max_sim_time, n_cluster_workers, memo_models, memo_degrees, stats_out, records_out,
                                          NULL, n_threads);
}
