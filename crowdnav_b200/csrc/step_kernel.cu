// step_kernel.cu -- one lockstep CrowdSim-v0 env-step for B environments (sm_100a).
//
// Replaces, for every env of the batch, crowd_sim/envs/crowd_sim.py:317-420 (CrowdSim.step, update=True):
//   N x Human.act -> ORCA.predict (orca.py:82-132, float32 RVO2 arithmetic, see orca_device.cuh),
//   optionally the robot's own ORCA.predict (explorer.py:42 with --policy orca),
//   robot-human swept-segment collision / min clearance (crowd_sim.py:331-351, utils.py:4-26), float64,
//   goal / timeout / reward ladder (crowd_sim.py:365-389), Euler integration (agent.py:122-135),
//   and Explorer.run_k_episodes' per-step bookkeeping (explorer.py:41-72).
//
// Mapping: one thread per (env, agent) -- L = N + 1 lanes per env (humans 0..N-1, lane N = robot), EPB envs per
// block, dense (an env's lanes may straddle a warp; all intra-env exchange goes through shared memory). Each lane
// loads its own agent with 16-byte loads (consecutive lanes -> consecutive addresses in the [B][N][2] arrays),
// stages it in shared memory for the other lanes' neighbour scans, solves its own ORCA problem, and writes its own
// agent back. HBM traffic per env-step is exactly the algorithmic 8*(19+12N)+2 bytes (+ episode bookkeeping).
#include "crowdsim_common.cuh"

namespace cs {

unsigned long long g_launches = 0;
int g_force_generic = 0;   // test hook: route every N through the generic one-thread-per-agent kernel

struct StepArgs {
    KParams k;
    int B, N, L, EPB;
    crowdsim_state st;
    crowdsim_step_io io;
    crowdsim_episodes ep;
    crowdsim_autoreset ar;
    int has_ep, has_ar;
    int act_only;      // crowdsim_orca_act: robot lanes solve and write action_out, nothing is mutated
    int n_steps;       // crowdsim_step_n: env-steps per launch (small-crowd kernel, ORCA robot)
    // crowdsim_onestep_lookahead (generic / crowd kernel only): step(action, update=False) -- outputs are written, the state is
    // not; the humans' next observable states go to la_pos / la_vel instead
    int lookahead;
    double *la_pos, *la_vel;
};

// ---- auto-reset protocol, consumer side (include/crowdsim_b200.h: crowdsim_autoreset) ----
// Robot lane: an env that just finished (or is parked waiting) looks at its next-scene slot. Returns 1 = install now.
// `s` = the slot state read (volatile) earlier in this launch: a slot the generator publishes later is simply picked
// up by the next step (the env parks for one step).
__device__ __forceinline__ int ar_decide(const StepArgs &A, int e, uint8_t s, bool finished, bool parked)
{
    if (!(finished || parked)) return 0;
    if (s == CROWDSIM_SLOT_READY) return 1;
    A.st.active[e] = 0;                                        // park: nothing to install (yet)
    A.ar.want[e] = (s == CROWDSIM_SLOT_EXHAUSTED) ? 0 : 1;
    return 0;
}
// Human lane a of env e: copy the prefetched scene into the live state (agent.py:47-58 set(px,py,gx,gy,0,0,...)).
// The generator published the slot with st.release; every lane that reads slot data acquires the flag first (and reads
// with ld.global.cg: L2 is the coherence point).
__device__ __forceinline__ void ar_install_human(const StepArgs &A, int e, int N, int a)
{
    const size_t i = (size_t)e * N + a;
    (void)ld_acquire_u8(A.ar.n_state + e);
    st2(A.st.h_pos, i, ld2_cg(A.ar.n_h_pos, i)); st2(A.st.h_vel, i, make_double2(0, 0));
    st2(A.st.h_goal, i, ld2_cg(A.ar.n_h_goal, i)); st2(A.st.h_attr, i, ld2_cg(A.ar.n_h_attr, i));
}
// Robot lane of env e: crowd_sim.py:262,274 (global_time = 0, robot.set(0,-R,0,R,0,0,pi/2)) + fresh episode accumulators.
__device__ __forceinline__ void ar_install_robot(const StepArgs &A, int e)
{
    (void)ld_acquire_u8(A.ar.n_state + e);
    st2(A.st.r_pos, e, make_double2(0.0, -A.ar.circle_radius)); st2(A.st.r_goal, e, make_double2(0.0, A.ar.circle_radius));
    st2(A.st.r_vel, e, make_double2(0, 0)); st2(A.st.r_attr, e, make_double2(A.ar.robot_radius, A.ar.robot_v_pref));
    if (A.st.r_theta) A.st.r_theta[e] = CS_PI / 2;
    A.st.g_time[e] = 0.0;
    if (A.has_ep) {
        A.ep.ep_steps[e] = 0; A.ep.ep_return[e] = 0.0; A.ep.ep_too_close[e] = 0; A.ep.ep_min_dist_sum[e] = 0.0;
        A.ep.ep_case[e] = __ldcg(A.ar.n_case + e);
    }
    A.st.active[e] = 1; A.ar.want[e] = 0;
}

}  // namespace cs
#include "step_flat.cuh"
#include "step_mid.cuh"
namespace cs {

// Resident blocks per SM the crowd kernel is compiled for. BASELINE config 4 (4096 envs x 21 agents = 683 blocks of 126
// threads) needs 5 per SM to be resident in ONE wave on 148 SMs; at 4 (119 registers) the launch ran 1.15 waves.
#ifndef CS_MID_MINBLOCKS
#define CS_MID_MINBLOCKS 5
#endif

// MID = false: the generic kernel of round 1 (RVO2's sequential code on per-thread shared-memory columns; any
// max_neighbors <= 10; kept as the A/B partner of the two fast kernels in the tests: crowdsim_debug_force_generic).
// MID = true: the crowd kernel for N > 5 (step_mid.cuh: register-resident lines, speculative LPs, compacted lp3).
// LIN: linear humans / robot (crowdsim_common.cuh: kLinHumans, kLinRobot), a compile-time choice as in step_flat_kernel.
template <bool MID, int LIN = 0>
__global__ void __launch_bounds__(MID ? 128 : 256, MID ? CS_MID_MINBLOCKS : 1) step_kernel(const __grid_constant__ StepArgs A)
{
    constexpr bool HLIN = (LIN & kLinHumans) != 0, RLIN = (LIN & kLinRobot) != 0;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_qcount;
    const int T = blockDim.x, tid = threadIdx.x;
    const int N = A.N, L = A.L;
    const KParams &k = A.k;
    const Stage s = carve_stage(smem, A.EPB, L, k.nb_alloc, T);
    if (MID && tid == 0) s_qcount = 0;

    const int le = tid / L, a = tid - le * L;
    const int e = blockIdx.x * A.EPB + le;
    const bool is_robot = (a == N);
    bool live = (e < A.B);
    if (live && A.st.active) live = (A.st.active[e] != 0);

    // ---- load own agent (coalesced 16-byte loads) and stage it ----
    double2 pos = make_double2(0, 0), vel = pos, goal = pos, attr = pos;
    double theta = 0, gtime = 0;
    if (live) {
        if (!is_robot) {
            const size_t i = (size_t)e * N + a;
            pos = ld2(A.st.h_pos, i); vel = ld2(A.st.h_vel, i); goal = ld2(A.st.h_goal, i); attr = ld2(A.st.h_attr, i);
        } else {
            pos = ld2(A.st.r_pos, e); vel = ld2(A.st.r_vel, e); goal = ld2(A.st.r_goal, e); attr = ld2(A.st.r_attr, e);
            gtime = A.st.g_time[e];
            if (k.robot_policy == CROWDSIM_ROBOT_EXTERNAL_ROT) theta = A.st.r_theta[e];
        }
    }
    stage_agent(s, k, tid, pos, vel, attr.x);
    __syncthreads();

    // ---- ORCA solves: every human lane; the robot lane iff the robot runs ORCA ----
    orca::V2 nv = orca::mk(0.f, 0.f);
    const bool solve = live && (!is_robot || k.robot_policy == CROWDSIM_ROBOT_ORCA) && !(A.act_only && !is_robot) && !(HLIN && !is_robot);
    if constexpr (LIN == (kLinHumans | kLinRobot)) (void)solve;      // nobody runs ORCA
    else if constexpr (MID) nv = mid_solve<kMidM>(s, k, solve, le, a, N, L, pos, goal, attr.y, tid, T, s.lines, &s_qcount);
    else if (solve) nv = orca_predict(s, k, le, a, N, L, pos, goal, attr.y, tid, T);

    if (A.act_only) {
        if (live && is_robot) st2(A.io.action_out, e, make_double2((double)nv.x, (double)nv.y));
        return;
    }

    // ---- robot lane publishes the velocity it applies this step ----
    double ax = 0, ay = 0;            // raw action: (vx, vy) or (v, r)
    double2 rvel = make_double2(0, 0); // world-frame velocity used by the collision test
    if (live && is_robot) {
        if constexpr (RLIN) { rvel = linear_velocity(pos, goal, attr.y); ax = rvel.x; ay = rvel.y; }
        else if (k.robot_policy == CROWDSIM_ROBOT_ORCA) { ax = (double)nv.x; ay = (double)nv.y; rvel = make_double2(ax, ay); }
        else {
            const double2 act = ld2(A.io.action, e); ax = act.x; ay = act.y;
            if (k.robot_policy == CROWDSIM_ROBOT_EXTERNAL_ROT) rvel = make_double2(ax * cos(ay + theta), ax * sin(ay + theta));  // crowd_sim.py:340-341
            else rvel = act;
        }
        s.act[le] = rvel;
    }
    __syncthreads();

    // ---- human lanes: swept-segment clearance against the robot (crowd_sim.py:333-345) ----
    const double dt = k.time_step;
    if (live && !is_robot) {
        const double2 rp = s.pos64[le * L + N], ra = s.act[le];
        const double px = pos.x - rp.x, py = pos.y - rp.y;
        const double vx = vel.x - ra.x, vy = vel.y - ra.y;     // human's CURRENT velocity attribute (previous action)
        const double ex = px + vx * dt, ey = py + vy * dt;
        s.closest[tid] = point_to_segment_dist0(px, py, ex, ey) - attr.x - s.rad64[le * L + N];
    }
    __syncthreads();

    // ---- robot lane: reduce clearances, ladder, update, bookkeeping; decides about auto-reset ----
    const bool env_ok = (e < A.B);
    int install = 0;
    if (is_robot && env_ok) {
        bool done = false;
        if (live) {
            double dmin = __longlong_as_double(0x7ff0000000000000LL); bool collision = false;
            for (int i = 0; i < N; ++i) {           // crowd_sim.py:346-351 (first collision breaks; dmin only matters without one)
                const double c = s.closest[le * L + i];
                if (c < 0) { collision = true; break; }
                else if (c < dmin) dmin = c;
            }
            double npx, npy, nvx, nvy;
            if (k.robot_policy != CROWDSIM_ROBOT_EXTERNAL_ROT) { npx = pos.x + ax * dt; npy = pos.y + ay * dt; nvx = ax; nvy = ay; }
            else { const double th = theta + ay; npx = pos.x + cos(th) * ax * dt; npy = pos.y + sin(th) * ax * dt; nvx = nvy = 0; }  // agent.py:115-118
            const bool reaching_goal = norm2(npx - goal.x, npy - goal.y) < attr.x;      // crowd_sim.py:365-366

            double reward; int info;                                                   // crowd_sim.py:368-389
            if (gtime >= k.time_limit - 1) { reward = 0; done = true; info = CROWDSIM_INFO_TIMEOUT; }
            else if (collision) { reward = k.collision_penalty; done = true; info = CROWDSIM_INFO_COLLISION; }
            else if (reaching_goal) { reward = k.success_reward; done = true; info = CROWDSIM_INFO_REACHGOAL; }
            else if (dmin < k.discomfort_dist) { reward = (dmin - k.discomfort_dist) * k.discomfort_penalty_factor * dt; done = false; info = CROWDSIM_INFO_DANGER; }
            else { reward = 0; done = false; info = CROWDSIM_INFO_NOTHING; }

            if (k.robot_policy == CROWDSIM_ROBOT_EXTERNAL_ROT) {                        // agent.py:133-135
                double nth = fmod(theta + ay, 2 * CS_PI); if (nth < 0) nth += 2 * CS_PI;
                if (!A.lookahead) A.st.r_theta[e] = nth;
                nvx = ax * cos(nth); nvy = ax * sin(nth);
            }
            const double ntime = gtime + dt;
            if (!A.lookahead) {
                st2(A.st.r_pos, e, make_double2(npx, npy));
                st2(A.st.r_vel, e, make_double2(nvx, nvy));
                A.st.g_time[e] = ntime;
            }
            if (A.io.action_out) st2(A.io.action_out, e, make_double2(nvx, nvy));
            A.io.reward[e] = reward; A.io.dmin[e] = dmin; A.io.done[e] = done ? 1 : 0; A.io.info[e] = (uint8_t)info;

            if (A.has_ep) {                                                            // explorer.py:41-72
                const crowdsim_episodes &ep = A.ep;
                const int t = ep.ep_steps[e];
                const double disc = (t < ep.discount_len) ? ep.discount[t] : 0.0;
                const double ret = ep.ep_return[e] + disc * reward;
                int tc = ep.ep_too_close[e]; double mds = ep.ep_min_dist_sum[e];
                if (info == CROWDSIM_INFO_DANGER) { tc += 1; mds += dmin; ep.ep_too_close[e] = tc; ep.ep_min_dist_sum[e] = mds; }
                ep.ep_return[e] = ret; ep.ep_steps[e] = t + 1;
                if (done) {
                    const int c = ep.ep_case[e];
                    if (c >= 0) {
                        ep.res_info[c] = (uint8_t)info; ep.res_steps[c] = t + 1;
                        ep.res_time[c] = (info == CROWDSIM_INFO_TIMEOUT) ? k.time_limit : ntime;
                        ep.res_return[c] = ret; ep.res_too_close[c] = tc; ep.res_min_dist_sum[c] = mds;
                        if (ep.res_final_rpos) st2(ep.res_final_rpos, c, make_double2(npx, npy));
                    }
                    if (A.st.active && !A.has_ar) A.st.active[e] = 0;
                }
            }
        }
        if (A.has_ar) install = ar_decide(A, e, ld_relaxed_u8(A.ar.n_state + e), live && done, !live && A.ar.want[e] != 0);
    }
    if (A.has_ar) {
        if (is_robot) s.closest[le * L + N] = (double)install;     // the robot's own clearance slot is unused: env-wide flag
        __syncthreads();
        install = (s.closest[le * L + N] != 0.0) && env_ok;
        if (install) {
            if (is_robot) ar_install_robot(A, e);
            else {
                ar_install_human(A, e, N, a);
                if (A.io.obs32) { const double2 np_ = ld2_cg(A.ar.n_h_pos, (size_t)e * N + a); reinterpret_cast<float4 *>(A.io.obs32)[(size_t)e * N + a] = make_float4((float)np_.x, (float)np_.y, 0.f, 0.f); }
            }
        }
        __syncthreads();
        if (install && is_robot) st_release_u8(A.ar.n_state + e, CROWDSIM_SLOT_EMPTY);
    }
    if (live && !is_robot && !install) {
        // agent.py:122-135 holonomic step with the ORCA action (float32 values widened) or the Linear action (float64)
        double hx = (double)nv.x, hy = (double)nv.y;
        if constexpr (HLIN) { const double2 lv = linear_human_velocity(pos, goal, attr.y); hx = lv.x; hy = lv.y; }
        const size_t i = (size_t)e * N + a;
        const double2 np_ = make_double2(pos.x + hx * dt, pos.y + hy * dt);
        if (A.lookahead) { st2(A.la_pos, i, np_); st2(A.la_vel, i, make_double2(hx, hy)); return; }   // agent.py:63-74, nothing mutated
        st2(A.st.h_pos, i, np_);
        st2(A.st.h_vel, i, make_double2(hx, hy));
        if (A.io.obs32) reinterpret_cast<float4 *>(A.io.obs32)[i] = make_float4((float)np_.x, (float)np_.y, HLIN ? (float)hx : nv.x, HLIN ? (float)hy : nv.y);
    }
}

// Packing of the small-crowd kernel is dense (32 / (N + 1) envs per warp). Sparser packings (fewer envs per warp) give
// more, less divergent warps, but were measured on B200 at 1 k .. 1 M envs and are never faster: the kernel's instruction
// stream is almost data-independent, so sparse warps only multiply the instruction count (profiles/r01_tune_epw_n5.txt).

// ---- crowdsim_orca_act for small crowds: the robot's ORCA decision only, ONE THREAD PER ENV. The step kernels' act_only mode
// runs the whole (env, agent) lane grid for the sake of the robot lanes (5 of 30 lanes useful); a host loop that asks for the
// robot's next decision after every step (batched.HostStepper) pays that second solve on every step. Same operations in the
// same order as the robot lane of step_flat_kernel (neighbour_order, make_line_sel, lp1_all, lp2_scan, lp3) => same result. ----
template <int N>
__global__ void __launch_bounds__(128) orca_act_kernel(const __grid_constant__ StepArgs A)
{
    using namespace orca;
    constexpr int M = N, T = 128;
    __shared__ float s_l[4 * M][T], s_pj[4 * M][T];          // per-thread line / projected-line columns for linearProgram3
    const int e = blockIdx.x * T + threadIdx.x, tid = threadIdx.x;
    if (e >= A.B) return;
    if (A.st.active && !A.st.active[e]) return;
    const KParams &k = A.k;
    const double2 pos = ld2(A.st.r_pos, e), vel = ld2(A.st.r_vel, e), goal = ld2(A.st.r_goal, e), attr = ld2(A.st.r_attr, e);
    const double gvx = goal.x - pos.x, gvy = goal.y - pos.y;
    const double speed = norm2(gvx, gvy);
    const V2 pref = mk((float)((speed > 1) ? gvx / speed : gvx), (float)((speed > 1) ? gvy / speed : gvy));
    const V2 p = mk((float)pos.x, (float)pos.y), v = mk((float)vel.x, (float)vel.y);
    const float r = (float)(attr.x + 0.01 + k.robot_safety_space), max_speed = (float)attr.y;
    V2 hp[M], hv[M]; float hr[M]; float dsq[M]; bool inr[M]; int id[M], src[M];
    #pragma unroll
    for (int c = 0; c < M; ++c) {
        const size_t i = (size_t)e * N + c;
        const double2 q = ld2(A.st.h_pos, i), w = ld2(A.st.h_vel, i), at = ld2(A.st.h_attr, i);
        hp[c] = mk((float)q.x, (float)q.y); hv[c] = mk((float)w.x, (float)w.y); hr[c] = (float)(at.x + 0.01 + k.robot_safety_space);
        dsq[c] = abssq(p - hp[c]); inr[c] = (k.max_neighbors > 0) && dsq[c] < sqr(k.neighbor_dist); id[c] = c;
    }
    int nl = neighbour_order<M>(dsq, inr, id, src);
    nl = nl < k.max_neighbors ? nl : k.max_neighbors;
    RegLines<M> R; bool valid[M];
    #pragma unroll
    for (int kk = 0; kk < M; ++kk) {
        valid[kk] = kk < nl; R.p[kk] = mk(0.f, 0.f); R.d[kk] = mk(0.f, 0.f);
        V2 qp = hp[0], qv = hv[0]; float qr = hr[0];
        #pragma unroll
        for (int c = 1; c < M; ++c) if (src[kk] == c) { qp = hp[c]; qv = hv[c]; qr = hr[c]; }
        if (valid[kk]) make_line_sel(p, v, r, qp, qv, qr, k.inv_time_horizon, k.inv_time_step, R.p[kk], R.d[kk]);
    }
    V2 cand[M]; bool feas[M];
    lp1_all<M, M>(R, valid, max_speed, pref, false, cand, feas);
    V2 nv = mk(0.f, 0.f);
    const int fail = lp2_scan<M, M>(R, valid, nl, cand, feas, lp2_init(pref, max_speed), nv);
    if (fail < nl) {
        const Lines Lr = { &s_l[0][tid], T }, Pr = { &s_pj[0][tid], T };
        #pragma unroll
        for (int kk = 0; kk < M; ++kk) Lr.set(kk, R.p[kk], R.d[kk]);
        lp3(Lr, nl, fail, max_speed, Pr, nv);
    }
    st2(A.io.action_out, e, make_double2((double)nv.x, (double)nv.y));
}

// SM count of the CURRENT device (cached per device: a process may drive several GPUs).
static int sm_count()
{
    static int cache[64];
    int dev = 0; cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    if (cache[dev] == 0) { int n = 0; cache[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148; }
    return cache[dev];
}

// n_steps launches of the crowd kernel (mid) or of the generic kernel for one policy combination
template <int LIN>
static int launch_crowd(const StepArgs &A, bool mid, int blocks, int threads, size_t smem, int n_steps, cudaStream_t stream)
{
    if (smem > 48 * 1024) {                                  // (a per-device attribute; setting it again is cheap)
        cudaError_t err = mid ? cudaFuncSetAttribute(step_kernel<true, LIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                              : cudaFuncSetAttribute(step_kernel<false, LIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return (int)err;
    }
    for (int rep = 0; rep < n_steps; ++rep) {
        if (mid) step_kernel<true, LIN><<<blocks, threads, smem, stream>>>(A);
        else step_kernel<false, LIN><<<blocks, threads, smem, stream>>>(A);
        ++g_launches;
    }
    return (int)cudaGetLastError();
}

static int launch(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, const crowdsim_step_io *io,
                  const crowdsim_episodes *ep, const crowdsim_autoreset *ar, int act_only, int n_steps, cudaStream_t stream,
                  double *la_pos = nullptr, double *la_vel = nullptr)
{
    if (!prm || !st || !io || B < 0 || N < 0 || n_steps < 1) return CROWDSIM_EINVAL;
    if (N > CROWDSIM_MAX_HUMANS || prm->max_neighbors > CROWDSIM_MAX_NEIGHBORS || !policies_supported(prm)) return CROWDSIM_EUNSUPPORTED;
    if (N > 0 && (!st->h_pos || !st->h_vel || !st->h_goal || !st->h_attr)) return CROWDSIM_EINVAL;
    if (!st->r_pos || !st->r_vel || !st->r_goal || !st->r_attr || !st->g_time) return CROWDSIM_EINVAL;
    if (prm->robot_policy == CROWDSIM_ROBOT_EXTERNAL_ROT && !st->r_theta) return CROWDSIM_EINVAL;
    if (act_only) { if (!io->action_out) return CROWDSIM_EINVAL; }
    else {
        if (!io->reward || !io->dmin || !io->done || !io->info) return CROWDSIM_EINVAL;
        if (prm->robot_policy != CROWDSIM_ROBOT_ORCA && prm->robot_policy != CROWDSIM_ROBOT_LINEAR && !io->action) return CROWDSIM_EINVAL;
    }
    if (ep && !act_only && (!ep->ep_case || !ep->ep_steps || !ep->ep_return || !ep->ep_too_close || !ep->ep_min_dist_sum ||
                            !ep->discount || !ep->res_info || !ep->res_steps || !ep->res_time || !ep->res_return ||
                            !ep->res_too_close || !ep->res_min_dist_sum)) return CROWDSIM_EINVAL;
    if (ar && !act_only) {
        if (!st->active || !ar->n_state || !ar->n_case || !ar->want || (N > 0 && (!ar->n_h_pos || !ar->n_h_goal || !ar->n_h_attr))) return CROWDSIM_EINVAL;
    }
    if (B == 0) return CROWDSIM_OK;
    StepArgs A;
    A.k = make_kparams(prm, N);
    if (act_only) A.k.robot_policy = CROWDSIM_ROBOT_ORCA;
    A.B = B; A.N = N; A.L = N + 1; A.EPB = envs_per_block(A.L, 128);
    A.st = *st; A.io = *io; A.has_ep = (ep != nullptr && !act_only); A.act_only = act_only; A.n_steps = 1;
    A.lookahead = (la_pos != nullptr); A.la_pos = la_pos; A.la_vel = la_vel;
    if (A.has_ep) A.ep = *ep; else memset(&A.ep, 0, sizeof(A.ep));
    A.has_ar = (ar != nullptr && !act_only);
    if (A.has_ar) A.ar = *ar; else memset(&A.ar, 0, sizeof(A.ar));
    const int lin = act_only ? 0 : lin_bits(prm);    // (orca_act: the robot's ORCA decision only, whatever the humans run)
    if (act_only && N >= 1 && N <= 5 && !g_force_generic) {
        const int blocks = (B + 127) / 128;
        switch (N) {
            case 1: orca_act_kernel<1><<<blocks, 128, 0, stream>>>(A); break;
            case 2: orca_act_kernel<2><<<blocks, 128, 0, stream>>>(A); break;
            case 3: orca_act_kernel<3><<<blocks, 128, 0, stream>>>(A); break;
            case 4: orca_act_kernel<4><<<blocks, 128, 0, stream>>>(A); break;
            default: orca_act_kernel<5><<<blocks, 128, 0, stream>>>(A); break;
        }
        ++g_launches;
        return (int)cudaGetLastError();
    }
    if (N >= 1 && N <= 5 && !g_force_generic && !A.lookahead) {
        // small crowds: register-resident solver, 32 / (N + 1) whole envs per warp (step_flat.cuh)
        const int epb = CS_FLAT_WPB * (32 / (N + 1));
        const int blocks = (B + epb - 1) / epb;
        const bool rot = A.k.robot_policy == CROWDSIM_ROBOT_EXTERNAL_ROT;
        // n steps in one launch with the state in registers: closed-loop only (the robot decides on device)
        const bool multi = n_steps > 1 && (A.k.robot_policy == CROWDSIM_ROBOT_ORCA || A.k.robot_policy == CROWDSIM_ROBOT_LINEAR);
        const int reps = multi ? 1 : n_steps;
        if (multi) A.n_steps = n_steps;
        // linearProgram3 queue of the single-step kernel: per warp when the launch leaves SMs mostly empty (latency-bound: no
        // block barrier, 2-4 % faster at 1 k - 4 k envs), per block when the chip is full (issue-bound: one warp runs the pass
        // for the whole block, 3-5 % faster at 64 k - 1 M envs). Measured with scripts/latency_probe.cu in round 1.
        const bool warpq = blocks * CS_FLAT_WPB <= 12 * sm_count();
        #define CS_FLAT_LAUNCH(NN, LN) do { if (multi) step_flat_kernel<NN, 99, false, true, true, LN><<<blocks, 32 * CS_FLAT_WPB, 0, stream>>>(A); \
                                            else if (rot) step_flat_kernel<NN, 99, !((LN) & kLinRobot), false, true, LN><<<blocks, 32 * CS_FLAT_WPB, 0, stream>>>(A); /* (never with a linear robot) */ \
                                            else if (warpq) step_flat_kernel<NN, 99, false, false, true, LN><<<blocks, 32 * CS_FLAT_WPB, 0, stream>>>(A); \
                                            else step_flat_kernel<NN, 99, false, false, false, LN><<<blocks, 32 * CS_FLAT_WPB, 0, stream>>>(A); } while (0)
        #define CS_FLAT_LAUNCH_N(NN) do { switch (lin) { case 0: CS_FLAT_LAUNCH(NN, 0); break; case 1: CS_FLAT_LAUNCH(NN, 1); break; \
                                                         case 2: CS_FLAT_LAUNCH(NN, 2); break; default: CS_FLAT_LAUNCH(NN, 3); break; } } while (0)
        for (int rep = 0; rep < reps; ++rep) {
            switch (N) {
                case 1: CS_FLAT_LAUNCH_N(1); break;
                case 2: CS_FLAT_LAUNCH_N(2); break;
                case 3: CS_FLAT_LAUNCH_N(3); break;
                case 4: CS_FLAT_LAUNCH_N(4); break;
                default: CS_FLAT_LAUNCH_N(5); break;
            }
            ++g_launches;
        }
        #undef CS_FLAT_LAUNCH_N
        #undef CS_FLAT_LAUNCH
        return (int)cudaGetLastError();
    }
    const int threads = A.EPB * A.L;
    const int blocks = (B + A.EPB - 1) / A.EPB;
    const bool mid = !g_force_generic && N > 5;              // (N = 0 and the forced A/B route stay on the generic kernel)
    const size_t smem = mid ? stage_bytes_mid(A.EPB, A.L, mid_lp3_floats()) : stage_bytes(A.EPB, A.L, A.k.nb_alloc, threads);
    switch (lin) {
        case 0: return launch_crowd<0>(A, mid, blocks, threads, smem, n_steps, stream);
        case 1: return launch_crowd<1>(A, mid, blocks, threads, smem, n_steps, stream);
        case 2: return launch_crowd<2>(A, mid, blocks, threads, smem, n_steps, stream);
        default: return launch_crowd<3>(A, mid, blocks, threads, smem, n_steps, stream);
    }
}

}  // namespace cs

extern "C" int crowdsim_step(const crowdsim_params *prm, int B, int N, crowdsim_state *st, crowdsim_step_io *io,
                             crowdsim_episodes *ep, const crowdsim_autoreset *ar, void *stream)
{
    return cs::launch(prm, B, N, st, io, ep, ar, 0, 1, (cudaStream_t)stream);
}

extern "C" int crowdsim_step_n(const crowdsim_params *prm, int B, int N, crowdsim_state *st, crowdsim_step_io *io,
                               crowdsim_episodes *ep, const crowdsim_autoreset *ar, int n_steps, void *stream)
{
    return cs::launch(prm, B, N, st, io, ep, ar, 0, n_steps, (cudaStream_t)stream);
}

extern "C" int crowdsim_onestep_lookahead(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, crowdsim_step_io *io,
                                          double *next_h_pos, double *next_h_vel, void *stream)
{
    if (!next_h_pos || !next_h_vel || !st) return CROWDSIM_EINVAL;
    if (io && io->obs32) return CROWDSIM_EINVAL;
    return cs::launch(prm, B, N, st, io, nullptr, nullptr, 0, 1, (cudaStream_t)stream, next_h_pos, next_h_vel);
}

extern "C" int crowdsim_orca_act(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, double *action_out,
                                 void *stream)
{
    crowdsim_step_io io; memset(&io, 0, sizeof(io)); io.action_out = action_out;
    return cs::launch(prm, B, N, st, &io, nullptr, nullptr, 1, 1, (cudaStream_t)stream);
}

extern "C" int crowdsim_graph_launch(void *graph_exec, void *stream, void *done_event)
{
    if (!graph_exec) return CROWDSIM_EINVAL;
    cudaError_t e = cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream);
    if (e == cudaSuccess && done_event) e = cudaEventRecord((cudaEvent_t)done_event, (cudaStream_t)stream);
    return (int)e;
}

extern "C" int crowdsim_host_pump(int n, void *const *graph_execs, void *const *graph_execs_alt, int alt_period, int first_round,
                                  void *const *streams, void *const *events,
                                  void *const *copy_dst, const void *const *copy_src, size_t copy_bytes, int rounds)
{
    // Round-robin over n independent batches (include/crowdsim_b200.h): wait for a batch's previous step, run the host-side
    // hand-over (copy_src -> copy_dst, e.g. "apply the decision the device computed"), enqueue its next step. The same loop
    // from an interpreter costs ~14 us per batch-step; here it is bounded by the copies and the launch call.
    if (n < 0 || rounds < 0 || !graph_execs || !streams || !events) return CROWDSIM_EINVAL;
    for (int r = 0; r < rounds; ++r)
        for (int i = 0; i < n; ++i) {
            cudaError_t e = cudaEventSynchronize((cudaEvent_t)events[i]);
            if (e != cudaSuccess) return (int)e;
            if (copy_bytes && copy_dst && copy_src && copy_dst[i] && copy_src[i]) memcpy(copy_dst[i], copy_src[i], copy_bytes);
            const bool alt = graph_execs_alt && alt_period > 1 && ((first_round + r) % alt_period) != 0;
            e = cudaGraphLaunch((cudaGraphExec_t)(alt ? graph_execs_alt[i] : graph_execs[i]), (cudaStream_t)streams[i]);
            if (e == cudaSuccess) e = cudaEventRecord((cudaEvent_t)events[i], (cudaStream_t)streams[i]);
            if (e != cudaSuccess) return (int)e;
        }
    return CROWDSIM_OK;
}

extern "C" int crowdsim_event_wait(void *event)
{
    if (!event) return CROWDSIM_EINVAL;
    return (int)cudaEventSynchronize((cudaEvent_t)event);
}

extern "C" void crowdsim_debug_force_generic(int on) { cs::g_force_generic = on; }

extern "C" int crowdsim_abi_version(void) { return CROWDSIM_ABI_VERSION; }

extern "C" unsigned long long crowdsim_launch_count(void) { return cs::g_launches; }

extern "C" int crowdsim_device_check(int *sm_count, int *cc_major, int *cc_minor)
{
    int dev = 0; cudaDeviceProp p;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&p, dev) != cudaSuccess) return CROWDSIM_ENODEVICE;
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return (p.major == 10) ? CROWDSIM_OK : CROWDSIM_ENODEVICE;
}
