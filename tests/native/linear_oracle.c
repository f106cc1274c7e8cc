/*
 * tests/native/linear_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The CPU oracle (oracle/crowdsim_oracle.c, included unchanged for its scenario generators, ORCA solve, segment test and
 * auto-reset) extended by crowdsim_params.human_policy and CROWDSIM_ROBOT_LINEAR: Linear.predict
 * (crowd_sim/envs/policy/linear.py:15-22) for the humans and / or the robot. Exports linear_oracle_step and
 * linear_oracle_lookahead_pack with the signatures of oracle_crowdsim_step / oracle_crowdsim_lookahead_pack; for ORCA humans
 * and an ORCA / external robot they compute exactly what those do.
 *
 * numpy's scalar np.arctan2 is within 1 ulp of C atan2 (np.cos / np.sin agree with glibc), so against the reference this path
 * is a tolerance, not bit-exactness. Build: gcc -O2 -ffp-contract=off -fopenmp (tests/linear_oracle.py).
 */
#include "../../oracle/crowdsim_oracle.c"

/* Linear.predict in float64. A human slot PARKED by rule `mixed` (include/crowdsim_b200.h) never moves; an agent standing on
 * its goal steps +x (atan2(0, 0) = 0) like the reference's. */
static void linear_predict(double px, double py, double gx, double gy, double v_pref, int parked_check, double *vx, double *vy)
{
    if (parked_check && px >= CROWDSIM_PARKED_X / 2) { *vx = 0.0; *vy = 0.0; return; }
    const double theta = atan2(gy - py, gx - px);
    *vx = cos(theta) * v_pref; *vy = sin(theta) * v_pref;
}

static int policies_supported(const crowdsim_params *p)
{
    return p->robot_policy >= CROWDSIM_ROBOT_EXTERNAL_XY && p->robot_policy <= CROWDSIM_ROBOT_LINEAR &&
           (p->human_policy == CROWDSIM_HUMANS_ORCA || p->human_policy == CROWDSIM_HUMANS_LINEAR);
}

/* crowd_sim.py:322-328 human actions, ORCA or Linear (env.config [humans] policy) */
static void human_actions(const crowdsim_params *p, int N, const double *hp, const double *hv, const double *hg, const double *ha,
                          const double *rp, const double *rv, const double *rg, const double *ra, double *hax, double *hay)
{
    for (int i = 0; i < N; ++i) {
        if (p->human_policy == CROWDSIM_HUMANS_LINEAR) {
            linear_predict(hp[2 * i], hp[2 * i + 1], hg[2 * i], hg[2 * i + 1], ha[2 * i + 1], 1, &hax[i], &hay[i]);
        } else {
            const orc_v2 a = orca_predict(p, N, hp, hv, hg, ha, rp, rv, rg, ra, i, NULL); hax[i] = a.x; hay[i] = a.y;
        }
    }
}

/* step_one of oracle/crowdsim_oracle.c with the policy choice: crowd_sim.py:317-420 (update=True) + explorer.py:41-72 */
static void lin_step_one(const crowdsim_params *p, int e, int N, crowdsim_state *st, crowdsim_step_io *io,
                         crowdsim_episodes *ep, const crowdsim_autoreset *ar)
{
    double *hp = st->h_pos + (size_t)e * N * 2, *hv = st->h_vel + (size_t)e * N * 2;
    const double *hg = st->h_goal + (size_t)e * N * 2, *ha = st->h_attr + (size_t)e * N * 2;
    double *rp = st->r_pos + 2 * e, *rv = st->r_vel + 2 * e; const double *rg = st->r_goal + 2 * e, *ra = st->r_attr + 2 * e;
    const double dt = p->time_step;
    double hax[CROWDSIM_MAX_HUMANS], hay[CROWDSIM_MAX_HUMANS];

    /* robot action first (explorer.py:42), from the same pre-update state */
    double ax, ay;
    if (p->robot_policy == CROWDSIM_ROBOT_ORCA) { const orc_v2 a = orca_predict(p, N, hp, hv, hg, ha, rp, rv, rg, ra, -1, NULL); ax = a.x; ay = a.y; }
    else if (p->robot_policy == CROWDSIM_ROBOT_LINEAR) linear_predict(rp[0], rp[1], rg[0], rg[1], ra[1], 0, &ax, &ay);
    else { ax = io->action[2 * e]; ay = io->action[2 * e + 1]; }
    human_actions(p, N, hp, hv, hg, ha, rp, rv, rg, ra, hax, hay);

    /* crowd_sim.py:331-351 collision / dmin; uses the humans' CURRENT velocity attribute (previous action) */
    const int rot = (p->robot_policy == CROWDSIM_ROBOT_EXTERNAL_ROT);
    double dmin = INFINITY; int collision = 0;
    for (int i = 0; i < N; ++i) {
        const double px = hp[2 * i] - rp[0], py = hp[2 * i + 1] - rp[1];
        double vx, vy;
        if (!rot) { vx = hv[2 * i] - ax; vy = hv[2 * i + 1] - ay; }
        else { vx = hv[2 * i] - ax * cos(ay + st->r_theta[e]); vy = hv[2 * i + 1] - ax * sin(ay + st->r_theta[e]); }
        const double ex = px + vx * dt, ey = py + vy * dt;
        const double closest = point_to_segment_dist0(px, py, ex, ey) - ha[2 * i] - ra[0];
        if (closest < 0) { collision = 1; break; }
        else if (closest < dmin) dmin = closest;
    }
    double npx, npy, ntheta, nvx, nvy;
    if (!rot) { npx = rp[0] + ax * dt; npy = rp[1] + ay * dt; nvx = ax; nvy = ay; }
    else { const double th = st->r_theta[e] + ay; npx = rp[0] + cos(th) * ax * dt; npy = rp[1] + sin(th) * ax * dt; nvx = nvy = 0; }
    const int reaching_goal = norm2(npx - rg[0], npy - rg[1]) < ra[0];

    double reward; int done, info;
    if (st->g_time[e] >= p->time_limit - 1) { reward = 0; done = 1; info = CROWDSIM_INFO_TIMEOUT; }
    else if (collision) { reward = p->collision_penalty; done = 1; info = CROWDSIM_INFO_COLLISION; }
    else if (reaching_goal) { reward = p->success_reward; done = 1; info = CROWDSIM_INFO_REACHGOAL; }
    else if (dmin < p->discomfort_dist) { reward = (dmin - p->discomfort_dist) * p->discomfort_penalty_factor * dt; done = 0; info = CROWDSIM_INFO_DANGER; }
    else { reward = 0; done = 0; info = CROWDSIM_INFO_NOTHING; }

    rp[0] = npx; rp[1] = npy;
    if (!rot) { rv[0] = nvx; rv[1] = nvy; }
    else { ntheta = fmod(st->r_theta[e] + ay, 2 * PI_D); if (ntheta < 0) ntheta += 2 * PI_D;
           st->r_theta[e] = ntheta; rv[0] = ax * cos(ntheta); rv[1] = ax * sin(ntheta); }
    for (int i = 0; i < N; ++i) { hp[2 * i] = hp[2 * i] + hax[i] * dt; hp[2 * i + 1] = hp[2 * i + 1] + hay[i] * dt; hv[2 * i] = hax[i]; hv[2 * i + 1] = hay[i]; }
    st->g_time[e] += dt;

    if (io->action_out) { io->action_out[2 * e] = rv[0]; io->action_out[2 * e + 1] = rv[1]; }
    io->reward[e] = reward; io->dmin[e] = dmin; io->done[e] = (uint8_t)done; io->info[e] = (uint8_t)info;

    if (ep) {
        const int t = ep->ep_steps[e];
        const double disc = (t < ep->discount_len) ? ep->discount[t] : 0.0;
        ep->ep_return[e] = ep->ep_return[e] + disc * reward;
        if (info == CROWDSIM_INFO_DANGER) { ep->ep_too_close[e] += 1; ep->ep_min_dist_sum[e] += dmin; }
        ep->ep_steps[e] = t + 1;
        if (done) {
            const int c = ep->ep_case[e];
            if (c >= 0) {
                ep->res_info[c] = (uint8_t)info; ep->res_steps[c] = t + 1;
                ep->res_time[c] = (info == CROWDSIM_INFO_TIMEOUT) ? p->time_limit : st->g_time[e];
                ep->res_return[c] = ep->ep_return[e]; ep->res_too_close[c] = ep->ep_too_close[e];
                ep->res_min_dist_sum[c] = ep->ep_min_dist_sum[e];
                if (ep->res_final_rpos) { ep->res_final_rpos[2 * c] = rp[0]; ep->res_final_rpos[2 * c + 1] = rp[1]; }
            }
            if (st->active && !ar) st->active[e] = 0;
        }
    }
    if (ar && done) autoreset_env(ar, e, N, st, ep);
}

int linear_oracle_step(const crowdsim_params *prm, int B, int N, crowdsim_state *st, crowdsim_step_io *io,
                       crowdsim_episodes *ep, const crowdsim_autoreset *ar)
{
    if (!prm || !st || !io || B < 0 || N < 0) return CROWDSIM_EINVAL;
    if (ar && !st->active) return CROWDSIM_EINVAL;
    if (N > CROWDSIM_MAX_HUMANS || prm->max_neighbors > CROWDSIM_MAX_NEIGHBORS || !policies_supported(prm)) return CROWDSIM_EUNSUPPORTED;
    #pragma omp parallel for schedule(static)
    for (int e = 0; e < B; ++e) {
        if (st->active && !st->active[e]) { if (ar && ar->want[e]) autoreset_env(ar, e, N, st, ep); continue; }
        lin_step_one(prm, e, N, st, io, ep, ar);
    }
    return 0;
}

/* oracle_crowdsim_lookahead_pack with the humans' policy: multi_human_rl.py:35-45, crowd_sim.py:314-315,414-416,
 * cadrl.py:104-129 (holonomic or unicycle robot actions, float32 rotate rows) */
int linear_oracle_lookahead_pack(const crowdsim_params *p, int B, int N, const crowdsim_state *st,
                                 const double *actions, int A, int unicycle, float *out_states, double *out_reward)
{
    if (!p || !st || !actions || !out_states || !out_reward) return CROWDSIM_EINVAL;
    if (!policies_supported(p)) return CROWDSIM_EUNSUPPORTED;
    const double dt = p->time_step;
    #pragma omp parallel for schedule(static)
    for (int e = 0; e < B; ++e) {
        const size_t o = (size_t)e * N * 2;
        const double *hp = st->h_pos + o, *hv = st->h_vel + o, *hg = st->h_goal + o, *ha = st->h_attr + o;
        const double *rp = st->r_pos + 2 * e, *rv = st->r_vel + 2 * e, *rg = st->r_goal + 2 * e, *ra = st->r_attr + 2 * e;
        double hax[CROWDSIM_MAX_HUMANS], hay[CROWDSIM_MAX_HUMANS];
        human_actions(p, N, hp, hv, hg, ha, rp, rv, rg, ra, hax, hay);
        for (int k = 0; k < A; ++k) {
            const double ax = actions[2 * k], ay = actions[2 * k + 1];
            double dmin = INFINITY; int collision = 0;
            for (int i = 0; i < N; ++i) {
                const double px = hp[2 * i] - rp[0], py = hp[2 * i + 1] - rp[1];
                double vx, vy;
                if (!unicycle) { vx = hv[2 * i] - ax; vy = hv[2 * i + 1] - ay; }
                else { vx = hv[2 * i] - ax * cos(ay + st->r_theta[e]); vy = hv[2 * i + 1] - ax * sin(ay + st->r_theta[e]); }
                const double ex = px + vx * dt, ey = py + vy * dt;
                const double closest = point_to_segment_dist0(px, py, ex, ey) - ha[2 * i] - ra[0];
                if (closest < 0) { collision = 1; break; } else if (closest < dmin) dmin = closest;
            }
            double npx, npy, nvx, nvy, nth;
            if (!unicycle) { npx = rp[0] + ax * dt; npy = rp[1] + ay * dt; nvx = ax; nvy = ay; nth = st->r_theta[e]; }
            else { nth = st->r_theta[e] + ay; nvx = ax * cos(nth); nvy = ax * sin(nth); npx = rp[0] + nvx * dt; npy = rp[1] + nvy * dt; }
            double gpx = npx, gpy = npy;
            if (unicycle) { const double th = st->r_theta[e] + ay; gpx = rp[0] + cos(th) * ax * dt; gpy = rp[1] + sin(th) * ax * dt; }
            const int reaching_goal = norm2(gpx - rg[0], gpy - rg[1]) < ra[0];
            double reward;
            if (st->g_time[e] >= p->time_limit - 1) reward = 0;
            else if (collision) reward = p->collision_penalty;
            else if (reaching_goal) reward = p->success_reward;
            else if (dmin < p->discomfort_dist) reward = (dmin - p->discomfort_dist) * p->discomfort_penalty_factor * dt;
            else reward = 0;
            out_reward[(size_t)e * A + k] = reward;
            for (int i = 0; i < N; ++i) {
                const double nhx = hp[2 * i] + hax[i] * dt, nhy = hp[2 * i + 1] + hay[i] * dt;
                float s[14] = { (float)npx, (float)npy, (float)nvx, (float)nvy, (float)ra[0], (float)rg[0], (float)rg[1], (float)ra[1],
                                (float)nth, (float)nhx, (float)nhy, (float)hax[i], (float)hay[i], (float)ha[2 * i] };
                rotate_row(s, unicycle, out_states + (((size_t)e * A + k) * N + i) * 13);
            }
        }
    }
    return 0;
}
