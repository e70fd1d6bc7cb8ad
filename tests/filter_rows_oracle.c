/*
 * filter_rows_oracle.c - TEST INFRASTRUCTURE: the C oracle's safety filter (oracle/lsm_oracle.c, compiled into this
 * translation unit unchanged) over independent rows, for tests/test_safety_filter_op.py.
 *
 * A row is one ego against M candidate others. It is run as a world of the ego (agent 0) and the row's active others
 * (agents 1.., in ascending slot order) through the oracle's own apply_safety_filter, whose result for agent 0 is the
 * row's result: np.argmin over the others in slot order, then the handle's resolution. Built by the test with the
 * oracle's compiler flags (no FMA contraction).
 */
#include "../oracle/lsm_oracle.c"

/* rel_form: 0 literal airtaxi relative position, 1 rotation form (lsmo_set_relative_state_form) */
static void row_world(env_t *w, const lsmo_params *p, const lsmo_grid *vg, int rel_form, double sep) {
    g_interp_f32 = (p->flags & LSMO_FLAG_INTERP_FLOAT32) != 0;
    g_rel_form = rel_form ? 1 : 0;
    w->p = p; w->vg = vg; w->dyn = p->dynamics;
    w->cur[9] = sep;
}

static void set_agent(env_t *w, int i, const double s[4]) {
    w->x[i] = s[0]; w->y[i] = s[1]; w->s2[i] = s[2]; w->s3[i] = s[3]; w->done[i] = 0;
}

/* safe_action [B][2]; filtered, index (deconflicting slot, -1 without an active slot), value (its HJ value, +inf without
 * one) [B]. Returns 0, or 1 on bad arguments (M + 1 above the oracle's agent limit, grid of the wrong dimensionality). */
int lsmt_safety_filter_rows(const lsmo_params *p, const lsmo_grid *vg, int rel_form, int64_t B, int32_t M, const double *ego,
                            const double *others, const double *ego_action, const double *other_actions,
                            const uint8_t *active, const double *separation_distance, double *safe_action,
                            uint8_t *filtered, int32_t *index, double *value) {
    if (vg == NULL || B < 0 || M < 0 || M + 1 > MAXN) return 1;
    if (vg->ndim != (p->dynamics == LSMO_DYN_DI ? 4 : 5)) return 1;
    env_t *w = (env_t *)calloc(1, sizeof(env_t));
    if (w == NULL) return 1;
    for (int64_t r = 0; r < B; ++r) {
        row_world(w, p, vg, rel_form, separation_distance ? separation_distance[r] : vg->separation_distance);
        double raw[MAXN][2], safe[MAXN][2];
        int filt[MAXN], deconf[MAXN], slot[MAXN], n = 1;
        set_agent(w, 0, ego + 4 * r);
        raw[0][0] = ego_action[2 * r]; raw[0][1] = ego_action[2 * r + 1];
        for (int k = 0; k < M; ++k) {
            const size_t s = (size_t)r * M + k;
            if (active && !active[s]) continue;
            set_agent(w, n, others + 4 * s);
            raw[n][0] = other_actions[2 * s]; raw[n][1] = other_actions[2 * s + 1];
            slot[n++] = k;
        }
        w->N = n;
        apply_safety_filter(w, raw, safe, filt, deconf);
        safe_action[2 * r] = safe[0][0]; safe_action[2 * r + 1] = safe[0][1];
        if (filtered) filtered[r] = (uint8_t)filt[0];
        if (index) index[r] = deconf[0] >= 1 ? slot[deconf[0]] : -1;
        if (value) {
            double v = INFINITY;
            if (deconf[0] >= 1) {       /* the minimum the filter selected: the deconflicting agent's value */
                double rel[5]; int inr;
                if (w->dyn == LSMO_DYN_DI) di_relative_state(w, 0, deconf[0], rel); else at_relative_state(w, 0, deconf[0], rel);
                v = hj_value(w, rel, &inr);
            }
            value[r] = v;
        }
    }
    free(w);
    return 0;
}

/* get_value_of_relative_state (+inf for NaN, shifted by -(sep - grid separation)) and the gradient components of K
 * relative states rel [K][d], or of the pairs (ego [K][4], other [K][4]) when rel is NULL. grad may be NULL. */
int lsmt_hj_lookup(const lsmo_params *p, const lsmo_grid *vg, int rel_form, int64_t K, const double *rel, const double *ego,
                   const double *other, const double *separation_distance, double *value, double *grad) {
    const int nd = p->dynamics == LSMO_DYN_DI ? 4 : 5;
    if (vg == NULL || K < 0 || vg->ndim != nd) return 1;
    env_t *w = (env_t *)calloc(1, sizeof(env_t));
    if (w == NULL) return 1;
    for (int64_t k = 0; k < K; ++k) {
        row_world(w, p, vg, rel_form, separation_distance ? separation_distance[k] : vg->separation_distance);
        double r[5];
        if (rel) for (int d = 0; d < nd; ++d) r[d] = rel[nd * k + d];
        else {
            set_agent(w, 0, ego + 4 * k); set_agent(w, 1, other + 4 * k); w->N = 2;
            if (w->dyn == LSMO_DYN_DI) di_relative_state(w, 0, 1, r); else at_relative_state(w, 0, 1, r);
        }
        int inr;
        value[k] = hj_value(w, r, &inr);
        if (grad) for (int d = 0; d < nd; ++d) grad[nd * k + d] = lsmo_interpolate(vg, r, d);
    }
    free(w);
    return 0;
}
