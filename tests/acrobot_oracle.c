/* acrobot_oracle.c -- the CPU oracle's discrete search with Acrobot-v1 as the env (test infrastructure).
 *
 * oracle/azg_oracle.c is the checker of the CartPole and Pendulum searches and stays as it is; this file includes it, so the network,
 * the head post-processing (softmax over the three logits), Philox / MT19937, the deterministic math, the selection (select_index:
 * epsilon-greedy, arg-max with random tie-break) and the value target are the oracle's own code.  What is new is the env (ac_step,
 * gym 0.17-0.19 classic_control/acrobot.py) and the discrete search loop and batch driver that step it: search_discrete_one /
 * worker / azo_search of the oracle with the env calls replaced and a 6-input network fed the observation of the node's hidden
 * state, line for line otherwise.  Node.r is the env's reward (-1.0 before the goal, 0.0 at it), terminal nodes get V = 0, the root
 * is never terminal.  The tree's state rows are the oracle's 4-wide rows, which hold the hidden state.
 *
 * Built by tests/acrobot_oracle.py with the flags of oracle/Makefile. */
#include "azg_oracle.c"

#define AC_WRAP_CAP 64 /* iterations per wrap loop, as ACROBOT_WRAP_CAP in the engine (env.cuh) */
#define AC_ERR_WRAP -4

static void ac_dsdt(const azo_config* c, const double* s, double a, double* d) {
    const double m1 = 1.0, m2 = 1.0, l1 = 1.0, lc1 = 0.5, lc2 = 0.5, I1 = 1.0, I2 = 1.0, g = 9.8, pi = 3.141592653589793;
    const double theta1 = s[0], theta2 = s[1], dtheta1 = s[2], dtheta2 = s[3];
    const double c2 = m_cos(c, theta2), s2 = m_sin(c, theta2);
    const double d1 = m1 * (lc1 * lc1) + m2 * (l1 * l1 + lc2 * lc2 + 2 * l1 * lc2 * c2) + I1 + I2;
    const double d2 = m2 * (lc2 * lc2 + l1 * lc2 * c2) + I2;
    const double phi2 = m2 * lc2 * g * m_cos(c, theta1 + theta2 - pi / 2.);
    const double phi1 = -m2 * l1 * lc2 * (dtheta2 * dtheta2) * s2 - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * s2 +
                        (m1 * lc1 + m2 * l1) * g * m_cos(c, theta1 - pi / 2) + phi2;
    const double ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * s2 - phi2) / (m2 * (lc2 * lc2) + I2 - (d2 * d2) / d1);
    const double ddtheta1 = -(d2 * ddtheta2 + phi1) / d1;
    d[0] = dtheta1; d[1] = dtheta2; d[2] = ddtheta1; d[3] = ddtheta2;
}

/* gym's wrap with each loop capped at AC_WRAP_CAP iterations (*capped = 1 when a loop would go on) */
static double ac_wrap(double x, int* capped) {
    const double pi = 3.141592653589793, diff = pi - -pi;
    for (int k = 0; x > pi; ++k) {
        if (k == AC_WRAP_CAP) { *capped = 1; return x; }
        x = x - diff;
    }
    for (int k = 0; x < -pi; ++k) {
        if (k == AC_WRAP_CAP) { *capped = 1; return x; }
        x = x + diff;
    }
    return x;
}

/* min(max(x, m), M) with Python's builtins: a NaN passes, -0 stays -0 */
static double ac_bound(double x, double m, double M) {
    x = m > x ? m : x;
    return M < x ? M : x;
}

/* one step: RK4 over [0, dt] of the book dynamics, wrap, bound; returns terminal, or AC_ERR_WRAP when a wrap loop reached its cap */
static int ac_step(const azo_config* c, const double* s, int action, double* o, double* reward) {
    const double dt = .2, pi = 3.141592653589793, MAX_VEL_1 = 4 * pi, MAX_VEL_2 = 9 * pi;
    const double torque = action == 0 ? -1.0 : (action == 1 ? 0.0 : 1.0);
    const double dt2 = dt / 2.0;
    double k1[4], k2[4], k3[4], k4[4], y[4];
    int capped = 0;
    ac_dsdt(c, s, torque, k1);
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt2 * k1[i];
    ac_dsdt(c, y, torque, k2);
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt2 * k2[i];
    ac_dsdt(c, y, torque, k3);
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt * k3[i];
    ac_dsdt(c, y, torque, k4);
    for (int i = 0; i < 4; ++i) o[i] = s[i] + dt / 6.0 * (k1[i] + 2 * k2[i] + 2 * k3[i] + k4[i]);
    o[0] = ac_wrap(o[0], &capped);
    o[1] = ac_wrap(o[1], &capped);
    o[2] = ac_bound(o[2], -MAX_VEL_1, MAX_VEL_1);
    o[3] = ac_bound(o[3], -MAX_VEL_2, MAX_VEL_2);
    const int terminal = -m_cos(c, o[0]) - m_cos(c, o[1] + o[0]) > 1.;
    *reward = terminal ? 0.0 : -1.0;
    return capped ? AC_ERR_WRAP : terminal;
}

/* _get_ob of a hidden state, each entry rounded to f32 */
static void ac_obs(const azo_config* c, const double* s, float* x) {
    x[0] = (float)m_cos(c, s[0]); x[1] = (float)m_sin(c, s[0]); x[2] = (float)m_cos(c, s[1]); x[3] = (float)m_sin(c, s[1]);
    x[4] = (float)s[2]; x[5] = (float)s[3];
}

void ac_observe(const azo_config* c, const double* s, float* obs) { ac_obs(c, s, obs); }

int ac_env_step(const azo_config* c, const double* s_in, int32_t action, double* s_out, double* reward, float* obs) {
    const int term = ac_step(c, s_in, action, s_out, reward);
    if (obs) ac_obs(c, s_out, obs);
    return term;
}

/* d_evaluate with the env's observation of the node's hidden state (6 entries) */
static void ac_evaluate(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, dtree_t* t, int node, int64_t* ctr) {
    const int A = t->A;
    float V, raw[AZO_MAX_A];
    if (c->use_eval_tape) {
        V = tp->V[b * t->R + node];
        for (int a = 0; a < A; ++a) t->prior[node * A + a] = tp->prior[(b * t->R + node) * A + a];
    } else {
        float x[6];
        ac_obs(c, t->state + node * 4, x);
        net_forward(net, c, x, &V, raw);
        azo_head_post(c, raw, t->prior + node * A);
        ctr[4]++;
    }
    t->V[node] = t->terminal[node] ? 0.0f : V;
    for (int a = 0; a < A; ++a) { t->eW[node * A + a] = 0.0; t->en[node * A + a] = 0; t->echild[node * A + a] = -1; }
}

/* search_discrete_one with the env's step; Node.r is the env's reward */
static int ac_search_one(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, const double* root_state, int32_t root_n,
                         dtree_t* t, rng_t* g, int64_t* ctr) {
    const int A = t->A;
    int err = 0;
    dtree_clear(t);
    t->n_nodes = 1;
    t->parent[0] = -1; t->paction[0] = -1; t->node_n[0] = root_n; t->terminal[0] = 0; t->r[0] = 0.0;
    for (int i = 0; i < 4; ++i) t->state[i] = root_state[i];
    ac_evaluate(c, net, tp, b, t, 0, ctr);
    for (int it = 0; it < c->n_rollouts; ++it) {
        int node = 0, created = 0;
        while (!t->terminal[node]) {
            double uct[AZO_MAX_A];
            double sq = sqrt((double)(t->node_n[node] + 1));
            for (int a = 0; a < A; ++a) {
                int n = t->en[node * A + a];
                double Q = n > 0 ? t->eW[node * A + a] / (double)n : (double)t->V[node];
                double pc = c->puct_f32 ? (double)(t->prior[node * A + a] * (float)c->c_uct) : (double)t->prior[node * A + a] * c->c_uct;
                uct[a] = Q + pc * (sq / (double)(n + 1));
            }
            int a = select_index(c, uct, A, g, &err);
            if (err) return err;
            ctr[1]++; ctr[2] += A;
            int child = t->echild[node * A + a];
            if (child >= 0) { node = child; continue; }
            child = t->n_nodes++;
            double rew;
            int term = ac_step(c, t->state + node * 4, a, t->state + child * 4, &rew);
            if (term == AC_ERR_WRAP) return AC_ERR_WRAP;
            t->parent[child] = node; t->paction[child] = a; t->node_n[child] = 0; t->terminal[child] = term; t->r[child] = rew;
            t->echild[node * A + a] = child;
            ac_evaluate(c, net, tp, b, t, child, ctr);
            node = child;
            created = 1;
            break;
        }
        if (!created) ctr[6]++; /* the trace ended on an existing terminal node: its return is backed up again */
        double R = (double)t->V[node];
        while (t->parent[node] >= 0) {
            R = t->r[node] + c->gamma * R;
            int p = t->parent[node], a = t->paction[node];
            t->en[p * A + a] += 1;
            t->eW[p * A + a] += R;
            node = p;
            t->node_n[node] += 1;
        }
        ctr[0]++;
    }
    return 0;
}

/* the discrete half of the oracle's worker */
static void* ac_worker(void* arg) {
    job_t* J = (job_t*)arg;
    const azo_config* cfg = J->cfg;
    const int R = azo_rows(cfg);
    const int A = cfg->num_actions;
    azo_results* res = J->res;
    dtree_t dt;
    dtree_alloc(&dt, R, A);
    for (;;) {
        int64_t b0 = __atomic_fetch_add(J->next, 16, __ATOMIC_RELAXED);
        if (b0 >= J->B) break;
        int64_t b1 = b0 + 16 < J->B ? b0 + 16 : J->B;
        for (int64_t b = b0; b < b1; ++b) {
            rng_t g;
            g.seed = cfg->seed; g.tree = J->tree_id0 + b; g.draws = 0; g.pw = 0; g.mt_mode = cfg->rng_mode == 1; g.mti = 624;
            if (g.mt_mode) mt_seed(&g, cfg->seed + (uint64_t)(J->tree_id0 + b));
            int e = ac_search_one(cfg, J->net, J->tapes, b, J->root_state + b * 4, J->root_n_init ? J->root_n_init[b] : 0, &dt, &g, J->ctr);
            if (!e && res) {
                double Q[AZO_MAX_A] = {0};
                res->n_children[b] = A;
                for (int a = 0; a < A; ++a) {
                    int n = dt.en[a];
                    Q[a] = n > 0 ? dt.eW[a] / (double)n : (double)dt.V[0];
                    res->actions[b * res->cmax + a] = (float)a;
                    res->counts[b * res->cmax + a] = n;
                    res->Q[b * res->cmax + a] = Q[a];
                }
                res->V_target[b] = value_target(cfg, Q, dt.en, A);
            }
            if (!e && J->dd) {
                azo_dump_discrete* dd = J->dd;
                dd->n_nodes[b] = dt.n_nodes;
                size_t o = (size_t)b * R;
                memcpy(dd->parent + o, dt.parent, R * 4); memcpy(dd->paction + o, dt.paction, R * 4);
                memcpy(dd->node_n + o, dt.node_n, R * 4); memcpy(dd->terminal + o, dt.terminal, R * 4);
                memcpy(dd->V + o, dt.V, R * 4); memcpy(dd->r + o, dt.r, R * 8);
                memcpy(dd->state + o * 4, dt.state, (size_t)R * 4 * 8);
                memcpy(dd->prior + o * A, dt.prior, (size_t)R * A * 4); memcpy(dd->eW + o * A, dt.eW, (size_t)R * A * 8);
                memcpy(dd->en + o * A, dt.en, (size_t)R * A * 4); memcpy(dd->echild + o * A, dt.echild, (size_t)R * A * 4);
            }
            J->ctr[5] += g.draws;
            if (e) __atomic_store_n(J->rc, e, __ATOMIC_RELAXED);
        }
    }
    dtree_free(&dt);
    return NULL;
}

/* azo_search for the discrete variant with num_actions 3 and state_dim 6 */
int ac_search(const azo_config* cfg, const float* weights, int64_t n_weights, int32_t B, const double* root_state, const int32_t* root_n_init,
              int64_t tree_id0, const azo_tapes* tapes, azo_results* res, azo_dump_discrete* dd, int32_t n_threads) {
    const int R = azo_rows(cfg);
    if (R > 4096 || cfg->hidden > 1024) return -2;
    if (cfg->variant != AZO_DISCRETE || cfg->num_actions != 3 || cfg->state_dim != 6) return -2;
    if (cfg->use_eval_tape && !tapes) return -2;
    net_t net;
    memset(&net, 0, sizeof net);
    if (!cfg->use_eval_tape && net_init(&net, cfg, weights, n_weights)) return -2;
    int rc = 0;
    int64_t next = 0;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    job_t jobs[256];
    pthread_t th[256];
    for (int i = 0; i < n_threads; ++i) {
        job_t j = {cfg, &net, tapes, root_state, root_n_init, tree_id0, B, res, dd, NULL, NULL, &next, &rc, {0}};
        jobs[i] = j;
    }
    for (int i = 1; i < n_threads; ++i) pthread_create(&th[i], NULL, ac_worker, &jobs[i]);
    ac_worker(&jobs[0]);
    for (int i = 1; i < n_threads; ++i) pthread_join(th[i], NULL);
    if (res && res->counters) {
        for (int k = 0; k < 8; ++k) res->counters[k] = 0;
        for (int i = 0; i < n_threads; ++i) for (int k = 0; k < 8; ++k) res->counters[k] += jobs[i].ctr[k];
    }
    if (!cfg->use_eval_tape) net_free(&net);
    return rc;
}
