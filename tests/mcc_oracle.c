/* mcc_oracle.c -- the CPU oracle's continuous search with MountainCarContinuous-v0 as the env (test infrastructure).
 *
 * oracle/azg_oracle.c is the checker of the Pendulum and CartPole searches and stays as it is; this file includes it, so the network,
 * the head post-processing, the action sampling, Philox / MT19937, the deterministic math, the selection and the value target are the
 * oracle's own code.  What is new is the env (mcc_step / mcc_obs, gym 0.17-0.19 classic_control/continuous_mountain_car.py) and the
 * continuous search loop and batch driver that step it: search_continuous_one / worker / azo_search of the oracle with the env calls
 * replaced, line for line otherwise.  The search reward is r / 16.2736044 as for every continuous search (mcts.py:687), terminal nodes
 * get V = 0, the root is never terminal.
 *
 * Built by tests/mcc_oracle.py with the flags of oracle/Makefile. */
#include "azg_oracle.c"

/* The f32 action enters f64 arithmetic exactly (numpy-1.x promotion); force = min(max(a, -1.0), 1.0) with Python's max / min (a NaN
 * passes, -0 stays -0); velocity + ((force * power) - (0.0025 * cos(3 * position))); the left wall sets velocity to +0; done =
 * position >= 0.45 and velocity >= 0; reward (done ? 100.0 : 0.0) - pow(a, 2) * 0.1 on the unclipped action (0 - x with the int 0 is
 * 0.0 - x: +0 for a zero action; pow(a, 2) of an f32 is exact in f64). */
static int mcc_step(const azo_config* c, const double* s, float action, double* o, double* reward) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.45, power = 0.0015;
    double pos = s[0], vel = s[1];
    const double a = (double)action;
    double force = -1.0 > a ? -1.0 : a;
    force = 1.0 < force ? 1.0 : force;
    vel = vel + (force * power - 0.0025 * m_cos(c, 3 * pos));
    if (vel > max_speed) vel = max_speed;
    if (vel < -max_speed) vel = -max_speed;
    pos = pos + vel;
    if (pos > max_position) pos = max_position;
    if (pos < min_position) pos = min_position;
    if (pos == min_position && vel < 0) vel = 0.0;
    const int done = pos >= goal_position && vel >= 0.0;
    *reward = (done ? 100.0 : 0.0) - (a * a) * 0.1;
    o[0] = pos; o[1] = vel;
    return done;
}

static void mcc_obs(const double* s, float* obs) {
    obs[0] = (float)s[0];
    obs[1] = (float)s[1];
}

int mcc_env_step(const azo_config* c, const double* s_in, float action, double* s_out, double* reward, float* obs) {
    const int term = mcc_step(c, s_in, action, s_out, reward);
    if (obs) mcc_obs(s_out, obs);
    return term;
}

/* c_evaluate with the env's observation */
static void mcc_evaluate(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, ctree_t* t, int row, int64_t* ctr) {
    float V;
    if (c->use_eval_tape) {
        V = tp->V[b * t->R + row];
    } else {
        float obs[2], raw[3 * AZO_MAX_K];
        mcc_obs(t->state + row * 2, obs);
        net_forward(net, c, obs, &V, raw);
        azo_head_post(c, raw, t->head + (size_t)row * t->K3);
        ctr[4]++;
    }
    t->V[row] = t->terminal[row] ? 0.0f : V;
}

/* search_continuous_one with the env's step */
static int mcc_search_one(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, const double* root_state, ctree_t* t,
                          rng_t* g, const int32_t* pw_table, int64_t* ctr) {
    int err = 0;
    int path[4096];
    ctree_clear(t);
    t->n_rows = 1;
    t->parent[0] = -1; t->expanded[0] = 1; t->node_n[0] = 0; t->terminal[0] = 0; t->r[0] = 0.0; t->en[0] = 0; t->eW[0] = 0.0;
    t->action[0] = 0.0f;
    t->state[0] = root_state[0]; t->state[1] = root_state[1];
    mcc_evaluate(c, net, tp, b, t, 0, ctr);
    c_add_pw_action(c, tp, b, t, 0, g, ctr);
    const float g32 = (float)c->gamma;
    for (int it = 0; it < c->n_rollouts; ++it) {
        int node = 0, depth = 0, created = 0;
        while (!t->terminal[node]) {
            int kids[4096], C = 0;
            for (int i = 1; i < t->n_rows; ++i) if (t->parent[i] == node) kids[C++] = i;
            int sel;
            if (pw_table[t->node_n[node]] - C > 0) {
                sel = c_add_pw_action(c, tp, b, t, node, g, ctr);
            } else {
                double uct[4096];
                double sq = sqrt((double)(t->node_n[node] + 1));
                for (int j = 0; j < C; ++j) {
                    int n = t->en[kids[j]];
                    double Q = n > 0 ? t->eW[kids[j]] / (double)n : (double)t->V[node];
                    uct[j] = Q + c->c_uct * (sq / (double)(n + 1));
                }
                sel = kids[select_index(c, uct, C, g, &err)];
                if (err) return err;
                ctr[2] += C;
            }
            ctr[1]++;
            path[depth++] = sel;
            if (t->expanded[sel]) { node = sel; continue; }
            double rew;
            int term = mcc_step(c, t->state + node * 2, t->action[sel], t->state + sel * 2, &rew);
            t->r[sel] = rew / PENDULUM_R_SCALE;
            t->terminal[sel] = term; t->expanded[sel] = 1; t->node_n[sel] = 0;
            mcc_evaluate(c, net, tp, b, t, sel, ctr);
            node = sel;
            created = 1;
            break;
        }
        if (!created) ctr[6]++;  /* the trace ended on an existing terminal node: its return is backed up again */
        double R = 0.0;
        for (int d = depth - 1; d >= 0; --d) {
            int row = path[d];
            if (d == depth - 1) R = t->r[row] + (double)(g32 * t->V[row]);
            else R = t->r[row] + c->gamma * R;
            t->en[row] += 1;
            t->eW[row] += R;
            t->node_n[t->parent[row]] += 1;
        }
        ctr[0]++;
    }
    return 0;
}

/* the continuous half of the oracle's worker */
static void* mcc_worker(void* arg) {
    job_t* J = (job_t*)arg;
    const azo_config* cfg = J->cfg;
    const int R = azo_rows(cfg);
    const int K = cfg->num_components, K3 = 3 * (K > 0 ? K : 1);
    azo_results* res = J->res;
    ctree_t ct;
    ctree_alloc(&ct, R, K3);
    for (;;) {
        int64_t b0 = __atomic_fetch_add(J->next, 16, __ATOMIC_RELAXED);
        if (b0 >= J->B) break;
        int64_t b1 = b0 + 16 < J->B ? b0 + 16 : J->B;
        for (int64_t b = b0; b < b1; ++b) {
            rng_t g;
            g.seed = cfg->seed; g.tree = J->tree_id0 + b; g.draws = 0; g.pw = 0; g.mt_mode = cfg->rng_mode == 1; g.mti = 624;
            if (g.mt_mode) {
                mt_seed(&g, cfg->seed + (uint64_t)(J->tree_id0 + b));
                torch_manual_seed(&g, cfg->seed + (uint64_t)(J->tree_id0 + b));
            }
            int e = mcc_search_one(cfg, J->net, J->tapes, b, J->root_state + b * 2, &ct, &g, J->pw_table, J->ctr);
            if (!e && res) {
                double Q[4096]; int32_t cnt[4096]; int C = 0;
                Q[0] = 0.0;
                for (int i = 1; i < ct.n_rows; ++i) if (ct.parent[i] == 0 && C < res->cmax) {
                    int n = ct.en[i];
                    Q[C] = n > 0 ? ct.eW[i] / (double)n : (double)ct.V[0];
                    cnt[C] = n;
                    res->actions[b * res->cmax + C] = ct.action[i];
                    res->counts[b * res->cmax + C] = n;
                    res->Q[b * res->cmax + C] = Q[C];
                    ++C;
                }
                res->n_children[b] = C;
                res->V_target[b] = value_target(cfg, Q, cnt, C);
            }
            if (!e && J->dc) {
                azo_dump_continuous* dc = J->dc;
                dc->n_rows[b] = ct.n_rows;
                size_t o = (size_t)b * R;
                memcpy(dc->parent + o, ct.parent, R * 4); memcpy(dc->action + o, ct.action, R * 4);
                memcpy(dc->eW + o, ct.eW, R * 8); memcpy(dc->en + o, ct.en, R * 4);
                memcpy(dc->expanded + o, ct.expanded, R * 4); memcpy(dc->node_n + o, ct.node_n, R * 4);
                memcpy(dc->terminal + o, ct.terminal, R * 4); memcpy(dc->V + o, ct.V, R * 4);
                memcpy(dc->r + o, ct.r, R * 8); memcpy(dc->state + o * 2, ct.state, (size_t)R * 2 * 8);
                memcpy(dc->head + o * K3, ct.head, (size_t)R * K3 * 4);
            }
            J->ctr[5] += g.draws;
            if (e) __atomic_store_n(J->rc, e, __ATOMIC_RELAXED);
        }
    }
    ctree_free(&ct);
    return NULL;
}

/* azo_search for the continuous variant with state_dim 2 */
int mcc_search(const azo_config* cfg, const float* weights, int64_t n_weights, int32_t B, const double* root_state, int64_t tree_id0,
               const azo_tapes* tapes, azo_results* res, azo_dump_continuous* dc, int32_t n_threads) {
    const int R = azo_rows(cfg);
    if (R > 4096 || cfg->hidden > 1024) return -2;
    if (cfg->variant != AZO_CONTINUOUS || cfg->state_dim != 2) return -2;
    if (cfg->num_components < 1 || cfg->num_components > AZO_MAX_K) return -2;
    if (cfg->use_eval_tape && !tapes) return -2;
    net_t net;
    memset(&net, 0, sizeof net);
    if (!cfg->use_eval_tape && net_init(&net, cfg, weights, n_weights)) return -2;
    int32_t* pw_table = malloc(sizeof(int32_t) * (cfg->n_rollouts + 2));
    for (int n = 0; n < cfg->n_rollouts + 2; ++n) pw_table[n] = azo_pw_limit(cfg->c_pw, cfg->kappa, n);
    int rc = 0;
    int64_t next = 0;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    job_t jobs[256];
    pthread_t th[256];
    for (int i = 0; i < n_threads; ++i) {
        job_t j = {cfg, &net, tapes, root_state, NULL, tree_id0, B, res, NULL, dc, pw_table, &next, &rc, {0}};
        jobs[i] = j;
    }
    for (int i = 1; i < n_threads; ++i) pthread_create(&th[i], NULL, mcc_worker, &jobs[i]);
    mcc_worker(&jobs[0]);
    for (int i = 1; i < n_threads; ++i) pthread_join(th[i], NULL);
    if (res && res->counters) {
        for (int k = 0; k < 8; ++k) res->counters[k] = 0;
        for (int i = 0; i < n_threads; ++i) for (int k = 0; k < 8; ++k) res->counters[k] += jobs[i].ctr[k];
    }
    free(pw_table);
    if (!cfg->use_eval_tape) net_free(&net);
    return rc;
}
