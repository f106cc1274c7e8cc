// step_flat.cuh -- CrowdSim step for small crowds (N <= 5 humans), register-resident ORCA solver, 1 .. n steps per launch.
//
// Same contract as step_kernel (crowd_sim/envs/crowd_sim.py:317-420 + orca.py:82-132 + explorer.py:41-72).
// Mapping: one thread per (env, agent) solve, L = N + 1 lanes per env, floor(32 / L) whole envs per warp so an env
// never straddles a warp: all intra-env exchange (candidate positions/velocities/radii for the neighbour scan, the
// robot's position and action for the swept-segment test, the per-human clearances for the min / any reduction) is
// done with warp shuffles -- no shared-memory staging, no block barrier on the common path.
// The <= N ORCA lines of a solve live in REGISTERS: every loop over lines is fully unrolled (template on N), so
// the LP code has static register indexing, no local/shared memory traffic and instruction-level parallelism
// across the independent (i, j) line pairs (speculative lp1 candidates + lp2 as a scan, orca_spec.cuh).
//
// linearProgram3 (needed by ~4.6 % of the solves, i.e. by some lane of ~3 of 4 warps) is NOT run in place: the
// solves that need it are compacted into a shared-memory queue. Inside linearProgram3 the sub-problem of each line i
// (linearProgram2 over the lines projected onto i, started from optVelocity * radius) depends only on the lines, not
// on the running result, so the <= N-1 sub-problems of a queued solve run on N-1 LANES IN PARALLEL (the sequential
// shared-memory LP code of orca_device.cuh), followed by a 4-step scan.
// The queue is per BLOCK (WARPQ = false: one warp runs the pass for the whole block, the others wait at a barrier;
// fewest instructions, best when the launch fills the chip) or per WARP (WARPQ = true: no block barrier, every warp runs
// the pass for its own 1-2 solves; best for launches that leave the SMs mostly empty). cs::launch() picks by grid size.
// Round 2 measured two finer splits of the pass, both bit-identical, both SLOWER, neither kept (profiles/r02_lp3_lanes.txt):
// (a) projections on (i, j) lanes + register-resident speculative sub-problems (orca_spec.cuh: lp3_project_pair /
// lp3_sub_spec, host-fuzzed): pass 4.4 vs 3.1 us at 4096 envs, 400 vs 162 us at 1 Mi envs; (b) four lane levels with
// early-exit code (projections, lp1 candidates, lp2 scans, outer scan; 10 lanes per item): 4.2 us / 195 us. More lanes
// per item means more warps with active lanes = more warp-instructions for the same work, and the all-pairs speculative
// form executes more instructions than early-exit code; at 1-2 warps per scheduler a warp's time is its instruction count.
//
// MULTI = true: crowdsim_step_n. With an ORCA robot nothing leaves the device between steps (explorer.py:41-43 is a pure
// loop), so a launch advances its envs n steps with the state in REGISTERS: one load of the state, n x (solve, collision,
// ladder, bookkeeping, install of the prefetched next scene when an episode ends), one store. That removes the launch gap
// and the load/store stage from every step but the first. Results are bit-identical to n x crowdsim_step.
//
// The multi-step kernel writes its memory effects once, at the end of the launch, from the registers; rare events (an
// episode's result row, parking, slot hand-over) are written when they happen. The single-step kernel stores as it goes.
#pragma once
#include "crowdsim_common.cuh"
#include "orca_spec.cuh"

namespace cs {

#define CS_FULL 0xffffffffu

// EPW = 32 / (N + 1) whole envs per warp (dense packing; sparser packings were measured and are never faster,
// profiles/r01_tune_epw_n5.txt). STAGE is a profiling aid (scripts/latency_probe.cu instantiates cut-down variants to
// attribute latency); the library only instantiates the full kernel (STAGE = 99).
// Register budget of the single-step kernel: 6 resident blocks per SM (<= 80 registers) is neutral at 4096 envs and 9 %
// faster at 65 k .. 1 M envs than the unconstrained build (round 1); the multi-step kernel serves launches that leave
// the chip mostly empty and carries ~35 registers of state across steps: 4 blocks per SM (<= 128 registers).
// Measured through bench.py (profiles/r02_multi_regs.txt): 3 / 4 / 5 blocks per SM = 131 / 128 / 96 registers give 790 / 848 /
// 878 M env-steps/s with 16 batches in flight and 390 / 399 / 389 M for a single batch: 4 is the balance.
// CS_FLAT_STRAIGHT_LINES (multi-step kernel): the M line constructions unconditionally and branch-free so that their chains
// interleave (profiles/r02_multi_straight_lines.txt: launch 72.9 -> 71.5 us); 0 = the branchy form of the single-step kernel.
// ROT: the robot is a unicycle (CROWDSIM_ROBOT_EXTERNAL_ROT, agent.py:115-135). A template parameter so that the double
// precision cos / sin / fmod code (12 % of the round-1 kernel's SASS) is only present in the kernels that execute it.
// LIN (kLinHumans | kLinRobot, crowdsim_common.cuh): humans and / or the robot follow Linear.predict (linear.py:15-22) instead
// of ORCA; selected at compile time like ROT, so the ORCA instantiations (LIN = 0) are the same code as without it.
#ifndef CS_FLAT_WPB
#define CS_FLAT_WPB 4
#endif
#ifndef CS_FLAT_MINBLOCKS
#define CS_FLAT_MINBLOCKS 6
#endif
#ifndef CS_FLAT_STRAIGHT_LINES
#define CS_FLAT_STRAIGHT_LINES 1
#endif
#ifndef CS_FLAT_MINBLOCKS_MULTI
#define CS_FLAT_MINBLOCKS_MULTI 4
#endif

template <int N, int STAGE = 99, bool ROT = false, bool MULTI = false, bool WARPQ = MULTI, int LIN = 0>
__global__ void __launch_bounds__(32 * CS_FLAT_WPB, (MULTI ? CS_FLAT_MINBLOCKS_MULTI : CS_FLAT_MINBLOCKS) * 4 / CS_FLAT_WPB)
step_flat_kernel(const __grid_constant__ StepArgs A)
{
    static_assert(STAGE == 99 || !MULTI, "stage cut-offs exist for the single-step kernel only");
    static_assert(!(ROT && MULTI), "a unicycle robot needs an external action every step");
    static_assert(WARPQ || !MULTI, "the multi-step kernel has no block barrier: warps run ahead of each other");
    static_assert(!(ROT && (LIN & kLinRobot)), "a linear robot is holonomic");
    constexpr bool HLIN = (LIN & kLinHumans) != 0, RLIN = (LIN & kLinRobot) != 0;
    if constexpr (STAGE == 0) return;
    using namespace orca;
    constexpr int L = N + 1, M = N, EPW = 32 / L, WPB = CS_FLAT_WPB;
    constexpr int T = 32 * WPB;
    constexpr int SUB = (M > 1) ? M - 1 : 1;                // lanes per queued lp3 item (sub-problems i = 1 .. M-1)
    constexpr int QF = 4 * M + 5;                           // floats per queued lp3 work item
    __shared__ float s_q[QF][T];                            // [field][slot]: lines of an item = orca::Lines(base = &s_q[0][slot], stride = T)
    __shared__ float s_p[4 * SUB][T];                       // per-thread projected lines of the sub-problem
    __shared__ float s_r2[3][T];                            // per-thread sub-problem result (x, y, ok)
    __shared__ float s_res[2][T];
    __shared__ int s_qcount;

    const KParams &k = A.k;
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    const int le = lane / L, a = lane - le * L;             // env within the warp, agent within the env
    const int ebase = le * L;                               // first lane of my env
    const int rl = ebase + N;                               // my env's robot lane
    const int e = (blockIdx.x * WPB + wib) * EPW + le;
    const bool is_robot = (a == N);
    const bool env_ok = (le < EPW) && (e < A.B);
    const size_t hi = (size_t)e * N + a;                    // my element of the [B][N][2] arrays (human lanes)
    if (!WARPQ && tid == 0) s_qcount = 0;

    // ---- all global loads of the launch are issued up front, unconditionally for valid envs, so that they overlap into ONE
    // DRAM round trip ----
    // (idle lanes get a goal 5 m away: a zero goal vector would drag the warp through the f64 sqrt / division slow paths)
    double2 pos = make_double2(0, 0), vel = pos, goal = make_double2(3, 4), attr = make_double2(0.3, 1.0);
    double theta = 0, gtime = 0; double2 ext = make_double2(0, 0);
    uint8_t act_flag = 1, slot_state = 0, want_flag = 0;
    int ep_t = 0, ep_tc = 0, ep_c = -1; double ep_ret = 0, ep_mds = 0;
    if (env_ok) {
        if (A.st.active) act_flag = A.st.active[e];
        if (!is_robot) {
            pos = ld2(A.st.h_pos, hi); vel = ld2(A.st.h_vel, hi); goal = ld2(A.st.h_goal, hi); attr = ld2(A.st.h_attr, hi);
        } else {
            pos = ld2(A.st.r_pos, e); vel = ld2(A.st.r_vel, e); goal = ld2(A.st.r_goal, e); attr = ld2(A.st.r_attr, e);
            gtime = A.st.g_time[e];
            if (ROT) theta = A.st.r_theta[e];
            if (!RLIN && k.robot_policy != CROWDSIM_ROBOT_ORCA) ext = ld2(A.io.action, e);
            if (A.has_ep) { ep_t = A.ep.ep_steps[e]; ep_ret = A.ep.ep_return[e]; ep_tc = A.ep.ep_too_close[e]; ep_mds = A.ep.ep_min_dist_sum[e]; ep_c = A.ep.ep_case[e]; }
            if (A.has_ar) { if (!MULTI) slot_state = ld_relaxed_u8(A.ar.n_state + e); want_flag = A.ar.want[e]; }
        }
    }
    if constexpr (STAGE == 1) {            // loads + stores only
        const bool live1 = env_ok && (act_flag != 0);
        if (live1 && !is_robot) { st2(A.st.h_pos, hi, pos); st2(A.st.h_vel, hi, make_double2(vel.x + goal.x * 0, vel.y + attr.x * 0)); }
        if (live1 && is_robot) { st2(A.st.r_pos, e, pos); A.st.g_time[e] = gtime + ext.x * 0 + theta * 0; }
        return;
    }

    // what this launch changed (decides the stores at the end)
    bool dirty_kin = false, dirty_scene = false, dirty_ep = false, any_live = false, new_case = false;
    double o_reward = 0, o_dmin = 0; double2 o_act = make_double2(0, 0); int o_done = 0, o_info = 0;
    const double dt = k.time_step;

    const int n_steps = MULTI ? A.n_steps : 1;
    #pragma unroll 1
    for (int s = 0; s < n_steps; ++s) {
    const bool live = env_ok && (act_flag != 0);
    if constexpr (MULTI) {
        // nothing left to do for this warp: every env is frozen and none is waiting for a scene
        if (__ballot_sync(CS_FULL, live || (is_robot && env_ok && want_flag != 0 && A.has_ar)) == 0u) break;
    }
    // float32 view of myself for the other lanes of my env (rvo2 boundary casts, orca.py:100-110)
    const float fpx = (float)pos.x, fpy = (float)pos.y, fvx = (float)vel.x, fvy = (float)vel.y;
    const float frh = (float)(attr.x + 0.01 + k.human_safety_space);     // my radius as seen by a human observer
    const float frr = (float)(attr.x + 0.01 + k.robot_safety_space);     // ... by the robot
    // (linear humans do not solve; with a linear robot too nobody does, and the solver below folds away)
    const bool solves = (LIN == (kLinHumans | kLinRobot)) ? false
                      : live && (!is_robot || k.robot_policy == CROWDSIM_ROBOT_ORCA) && !(HLIN && !is_robot);

    // ---- orca.py:113-115 preferred velocity (float64) ----
    const double gvx = goal.x - pos.x, gvy = goal.y - pos.y;
    const double speed = norm2(gvx, gvy);
    const V2 pref = mk((float)((speed > 1) ? gvx / speed : gvx), (float)((speed > 1) ? gvy / speed : gvy));
    const V2 p = mk(fpx, fpy), v = mk(fvx, fvy);
    const float r = is_robot ? frr : frh;
    const float max_speed = (float)attr.y;

    // ---- neighbour scan: candidate slot c -> agent j (reference order: other humans, then the robot iff visible) ----
    float dsq[M]; bool inr[M]; int jj[M];
    #pragma unroll
    for (int c = 0; c < M; ++c) {
        int j; bool cv;
        if (is_robot) { j = c; cv = true; }
        else if (c < N - 1) { j = (c < a) ? c : c + 1; cv = true; }
        else { j = N; cv = (k.robot_visible != 0); }
        jj[c] = j;
        const float qx = __shfl_sync(CS_FULL, fpx, ebase + j), qy = __shfl_sync(CS_FULL, fpy, ebase + j);
        dsq[c] = abssq(p - mk(qx, qy));
        inr[c] = solves && cv && (k.max_neighbors > 0) && dsq[c] < sqr(k.neighbor_dist);
    }
    // rank of each candidate = position RVO2's insertion sort (strict <, ties in scan order) would give it: for cc < c,
    // cc precedes c iff dsq[cc] <= dsq[c] -- one comparison per unordered pair. The agent index of the kk-th nearest is
    // then read from a packed word (3 bits per position, N <= 5) instead of an M x M select cascade (orca_spec.cuh:
    // neighbour_order is the host-checked copy of these statements).
    int rank[M];
    #pragma unroll
    for (int c = 0; c < M; ++c) rank[c] = 0;
    #pragma unroll
    for (int c = 1; c < M; ++c) {
        #pragma unroll
        for (int cc = 0; cc < c; ++cc) {
            const bool le_ = dsq[cc] <= dsq[c];
            rank[c] += (inr[cc] && le_) ? 1 : 0;
            rank[cc] += (inr[c] && !le_) ? 1 : 0;
        }
    }
    int nl = 0; unsigned packed = 0u;
    #pragma unroll
    for (int c = 0; c < M; ++c) if (inr[c]) { packed |= (unsigned)jj[c] << (3 * rank[c]); ++nl; }
    int src[M];                             // src[kk] = agent index of the kk-th nearest (0 beyond nl)
    #pragma unroll
    for (int kk = 0; kk < M; ++kk) src[kk] = (int)((packed >> (3 * kk)) & 7u);
    nl = nl < k.max_neighbors ? nl : k.max_neighbors;

    // ---- ORCA lines in rank order, in registers ----
    RegLines<M> R; bool valid[M];
    if constexpr (CS_FLAT_STRAIGHT_LINES && MULTI) {
        // multi-step kernel (1-2 warps per scheduler: a launch lasts as long as one warp's dependent chains): all M constructions
        // unconditionally and branch-free, so that their chains interleave; absent positions get a far-away dummy neighbour (no
        // special values) and are zeroed afterwards, the rare overlapping lines (0.09 %) are repaired behind a warp vote.
        V2 qp[M], qv[M]; float qr[M]; bool ov[M]; bool any_ov = false;
        #pragma unroll
        for (int kk = 0; kk < M; ++kk) {
            const int sl = ebase + src[kk];
            const float qx = __shfl_sync(CS_FULL, fpx, sl), qy = __shfl_sync(CS_FULL, fpy, sl);
            const float wx = __shfl_sync(CS_FULL, fvx, sl), wy = __shfl_sync(CS_FULL, fvy, sl);
            const float rh = __shfl_sync(CS_FULL, frh, sl), rr = __shfl_sync(CS_FULL, frr, sl);
            valid[kk] = kk < nl;
            qp[kk] = valid[kk] ? mk(qx, qy) : mk(fpx + 100.0f, fpy); qv[kk] = valid[kk] ? mk(wx, wy) : mk(0.f, 0.f);
            qr[kk] = valid[kk] ? (is_robot ? rr : rh) : r;
        }
        #pragma unroll
        for (int kk = 0; kk < M; ++kk) {
            make_line_far(p, v, r, qp[kk], qv[kk], qr[kk], k.inv_time_horizon, R.p[kk], R.d[kk], ov[kk]);
            ov[kk] = ov[kk] && valid[kk]; any_ov = any_ov || ov[kk];
        }
        if (__any_sync(CS_FULL, any_ov)) {
            #pragma unroll
            for (int kk = 0; kk < M; ++kk) if (ov[kk]) make_line_overlap(p, v, r, qp[kk], qv[kk], qr[kk], k.inv_time_step, R.p[kk], R.d[kk]);
        }
        #pragma unroll
        for (int kk = 0; kk < M; ++kk) if (!valid[kk]) { R.p[kk] = mk(0.f, 0.f); R.d[kk] = mk(0.f, 0.f); }
    } else {
    #pragma unroll
    for (int kk = 0; kk < M; ++kk) {
        const int sl = ebase + src[kk];
        const float qx = __shfl_sync(CS_FULL, fpx, sl), qy = __shfl_sync(CS_FULL, fpy, sl);
        const float wx = __shfl_sync(CS_FULL, fvx, sl), wy = __shfl_sync(CS_FULL, fvy, sl);
        const float rh = __shfl_sync(CS_FULL, frh, sl), rr = __shfl_sync(CS_FULL, frr, sl);
        valid[kk] = kk < nl;
        R.p[kk] = mk(0.f, 0.f); R.d[kk] = mk(0.f, 0.f);
        if (valid[kk]) make_line_sel(p, v, r, mk(qx, qy), mk(wx, wy), is_robot ? rr : rh, k.inv_time_horizon, k.inv_time_step, R.p[kk], R.d[kk]);
    }
    }
    if constexpr (STAGE == 2) {            // + preferred velocity, neighbour scan, ORCA lines
        float acc = pref.x + pref.y;
        #pragma unroll
        for (int kk = 0; kk < M; ++kk) acc += R.p[kk].x + R.p[kk].y + R.d[kk].x + R.d[kk].y;
        if (live && !is_robot) st2(A.st.h_vel, hi, make_double2(vel.x, vel.y + (double)acc * 0));
        return;
    }

    // ---- linear programs: speculative lp1 candidates for every line (orca_spec.cuh), then linearProgram2 as a scan ----
    V2 cand[M]; bool feas[M];
    lp1_all<M, M>(R, valid, max_speed, pref, false, cand, feas);
    V2 nv = mk(0.f, 0.f);
    const int fail = lp2_scan<M, M>(R, valid, nl, cand, feas, lp2_init(pref, max_speed), nv);
    if constexpr (STAGE == 3) {            // + lp1 candidates and the lp2 scan
        if (live && !is_robot) st2(A.st.h_vel, hi, make_double2(vel.x + (double)nv.x * 0, vel.y + (double)(nv.y + fail) * 0));
        return;
    }

    // ---- linearProgram3: the solves that need it are compacted into a shared-memory queue; the sub-problems of an item
    // run on SUB lanes in parallel (sequential shared-memory LP code of orca_device.cuh), one lane finishes with
    // linearProgram3's outer scan ----
    const bool need3 = solves && fail < nl;
    if constexpr (WARPQ) {
        // warp-level queue: no block barrier; every warp runs the sub-problems of its own solves
        const unsigned m3 = __ballot_sync(CS_FULL, need3);
        if (m3) {
            const int wbase = wib * 32;
            const int cnt = __popc(m3);
            const int slot = wbase + __popc(m3 & ((1u << lane) - 1u));
            if (need3) {
                #pragma unroll
                for (int kk = 0; kk < M; ++kk) {
                    s_q[4 * kk + 0][slot] = R.p[kk].x; s_q[4 * kk + 1][slot] = R.p[kk].y;
                    s_q[4 * kk + 2][slot] = R.d[kk].x; s_q[4 * kk + 3][slot] = R.d[kk].y;
                }
                s_q[4 * M + 0][slot] = __int_as_float(nl); s_q[4 * M + 1][slot] = __int_as_float(fail);
                s_q[4 * M + 2][slot] = max_speed; s_q[4 * M + 3][slot] = nv.x; s_q[4 * M + 4][slot] = nv.y;
            }
            __syncwarp();
            constexpr int IPP = 32 / SUB;                        // items per pass
            for (int base = 0; base < cnt; base += IPP) {
                const int item = wbase + base + lane / SUB, i = lane % SUB + 1;
                const bool mine = (lane < IPP * SUB) && (base + lane / SUB) < cnt;
                if (mine) {
                    const Lines Lq = { &s_q[0][item], T };
                    const int qn = __float_as_int(s_q[4 * M + 0][item]);
                    bool ok = false; V2 r2 = mk(0.f, 0.f);
                    if (M > 1 && i < qn) {
                        const Lines Pq = { &s_p[0][tid], T };
                        ok = lp3_subproblem(Lq, i, s_q[4 * M + 2][item], Pq, r2);
                    }
                    s_r2[0][tid] = r2.x; s_r2[1][tid] = r2.y; s_r2[2][tid] = ok ? 1.0f : 0.0f;
                }
                __syncwarp();
                if (mine && i == 1) {
                    const Lines Lq = { &s_q[0][item], T };
                    const int qn = __float_as_int(s_q[4 * M + 0][item]), qf = __float_as_int(s_q[4 * M + 1][item]);
                    const float qr = s_q[4 * M + 2][item];
                    V2 res = mk(s_q[4 * M + 3][item], s_q[4 * M + 4][item]);
                    lp3_outer_scan(Lq, qn, qf, qr, res, [&](int ii, V2 &r2) {
                        const int src_ = tid + (ii - 1);
                        r2 = mk(s_r2[0][src_], s_r2[1][src_]);
                        return s_r2[2][src_] != 0.0f;
                    });
                    s_res[0][item] = res.x; s_res[1][item] = res.y;
                }
                __syncwarp();
            }
            if (need3) nv = mk(s_res[0][slot], s_res[1][slot]);
            __syncwarp();                                        // the queue is reused by the next step (MULTI)
        }
    } else {
        __syncthreads();                                         // s_qcount = 0 visible
        int slot = -1;
        if (need3) {
            slot = atomicAdd(&s_qcount, 1);
            #pragma unroll
            for (int kk = 0; kk < M; ++kk) {
                s_q[4 * kk + 0][slot] = R.p[kk].x; s_q[4 * kk + 1][slot] = R.p[kk].y;
                s_q[4 * kk + 2][slot] = R.d[kk].x; s_q[4 * kk + 3][slot] = R.d[kk].y;
            }
            s_q[4 * M + 0][slot] = __int_as_float(nl); s_q[4 * M + 1][slot] = __int_as_float(fail);
            s_q[4 * M + 2][slot] = max_speed; s_q[4 * M + 3][slot] = nv.x; s_q[4 * M + 4][slot] = nv.y;
        }
        if (__syncthreads_or(need3 ? 1 : 0)) {
            const int cnt = s_qcount;
            constexpr int IPP = T / SUB;                         // items per pass
            for (int base = 0; base < cnt; base += IPP) {
                const int item = base + tid / SUB, i = tid % SUB + 1;
                const bool mine = (tid < IPP * SUB) && item < cnt;
                if (mine) {
                    const Lines Lq = { &s_q[0][item], T };
                    const int qn = __float_as_int(s_q[4 * M + 0][item]);
                    bool ok = false; V2 r2 = mk(0.f, 0.f);
                    if (M > 1 && i < qn) {
                        // sequential shared-memory LP code with early exits: measured faster here than every finer or
                        // speculative split tried (header; profiles/r02_lp3_lanes.txt)
                        const Lines Pq = { &s_p[0][tid], T };
                        ok = lp3_subproblem(Lq, i, s_q[4 * M + 2][item], Pq, r2);
                    }
                    s_r2[0][tid] = r2.x; s_r2[1][tid] = r2.y; s_r2[2][tid] = ok ? 1.0f : 0.0f;
                }
                __syncthreads();
                if (mine && i == 1) {                            // the item's first lane runs linearProgram3's outer scan
                    const Lines Lq = { &s_q[0][item], T };
                    const int qn = __float_as_int(s_q[4 * M + 0][item]), qf = __float_as_int(s_q[4 * M + 1][item]);
                    const float qr = s_q[4 * M + 2][item];
                    V2 res = mk(s_q[4 * M + 3][item], s_q[4 * M + 4][item]);
                    lp3_outer_scan(Lq, qn, qf, qr, res, [&](int ii, V2 &r2) {
                        const int src_ = tid + (ii - 1);              // lane of sub-problem ii of this item
                        r2 = mk(s_r2[0][src_], s_r2[1][src_]);
                        return s_r2[2][src_] != 0.0f;
                    });
                    s_res[0][item] = res.x; s_res[1][item] = res.y;
                }
                __syncthreads();
            }
            if (need3) nv = mk(s_res[0][slot], s_res[1][slot]);
        }
    }

    if constexpr (STAGE == 4) {            // + lp3
        if (live && !is_robot) st2(A.st.h_vel, hi, make_double2(vel.x + (double)nv.x * 0, vel.y + (double)nv.y * 0));
        return;
    }
    // ---- robot velocity of this step, broadcast inside the env ----
    double ax = 0, ay = 0, rvx = 0, rvy = 0;
    if (is_robot) {
        if constexpr (RLIN) { const double2 lv = linear_velocity(pos, goal, attr.y); ax = lv.x; ay = lv.y; rvx = ax; rvy = ay; }
        else if (k.robot_policy == CROWDSIM_ROBOT_ORCA) { ax = (double)nv.x; ay = (double)nv.y; rvx = ax; rvy = ay; }
        else if (ROT) { ax = ext.x; ay = ext.y; rvx = ax * cos(ay + theta); rvy = ax * sin(ay + theta); }      // crowd_sim.py:340-341
        else { ax = ext.x; ay = ext.y; rvx = ax; rvy = ay; }
    }
    const double Rvx = __shfl_sync(CS_FULL, rvx, rl), Rvy = __shfl_sync(CS_FULL, rvy, rl);
    const double Rpx = __shfl_sync(CS_FULL, pos.x, rl), Rpy = __shfl_sync(CS_FULL, pos.y, rl);
    const double Rrad = __shfl_sync(CS_FULL, attr.x, rl);

    // ---- human lanes: swept-segment clearance (crowd_sim.py:333-345) ----
    double closest = 0.0;
    if (live && !is_robot) {
        const double px = pos.x - Rpx, py = pos.y - Rpy;
        const double vx = vel.x - Rvx, vy = vel.y - Rvy;    // the human's CURRENT velocity attribute (previous action)
        const double ex = px + vx * dt, ey = py + vy * dt;
        closest = point_to_segment_dist0(px, py, ex, ey) - attr.x - Rrad;
    }
    // ordered fold over the env's humans (first collision breaks, crowd_sim.py:346-351); consumed by the robot lane
    double dmin = __longlong_as_double(0x7ff0000000000000LL); bool collision = false;
    #pragma unroll
    for (int i = 0; i < N; ++i) {
        const double ci = __shfl_sync(CS_FULL, closest, ebase + i);
        if (!collision) { if (ci < 0) collision = true; else if (ci < dmin) dmin = ci; }
    }

    // ---- robot lane: ladder (crowd_sim.py:365-389), update (agent.py:110-135), bookkeeping (explorer.py:41-72);
    // decides about auto-reset ----
    int install = 0;
    if (is_robot && env_ok) {
        bool done = false;
        if (live) {
            double npx, npy, nvx, nvy;
            if (!ROT) { npx = pos.x + ax * dt; npy = pos.y + ay * dt; nvx = ax; nvy = ay; }
            else { const double th = theta + ay; npx = pos.x + cos(th) * ax * dt; npy = pos.y + sin(th) * ax * dt; nvx = nvy = 0; }
            const bool reaching_goal = norm2(npx - goal.x, npy - goal.y) < attr.x;
            double reward; int info;
            if (gtime >= k.time_limit - 1) { reward = 0; done = true; info = CROWDSIM_INFO_TIMEOUT; }
            else if (collision) { reward = k.collision_penalty; done = true; info = CROWDSIM_INFO_COLLISION; }
            else if (reaching_goal) { reward = k.success_reward; done = true; info = CROWDSIM_INFO_REACHGOAL; }
            else if (dmin < k.discomfort_dist) { reward = (dmin - k.discomfort_dist) * k.discomfort_penalty_factor * dt; done = false; info = CROWDSIM_INFO_DANGER; }
            else { reward = 0; done = false; info = CROWDSIM_INFO_NOTHING; }
            if (ROT) {                                                                   // agent.py:133-135
                double nth = fmod(theta + ay, 2 * CS_PI); if (nth < 0) nth += 2 * CS_PI;
                theta = nth; nvx = ax * cos(nth); nvy = ax * sin(nth);
            }
            pos = make_double2(npx, npy); vel = make_double2(nvx, nvy);
            gtime = gtime + dt;
            if constexpr (MULTI) { o_act = vel; o_reward = reward; o_dmin = dmin; o_done = done ? 1 : 0; o_info = info; any_live = true; dirty_kin = true; }
            else {                                           // single step: nothing to carry, state and outputs leave at once
                st2(A.st.r_pos, e, pos); st2(A.st.r_vel, e, vel); A.st.g_time[e] = gtime; if (ROT) A.st.r_theta[e] = theta;
                if (A.io.action_out) st2(A.io.action_out, e, vel);
                A.io.reward[e] = reward; A.io.dmin[e] = dmin; A.io.done[e] = done ? 1 : 0; A.io.info[e] = (uint8_t)info;
            }
            if (A.has_ep) {
                const crowdsim_episodes &ep = A.ep;
                const double disc = (ep_t < ep.discount_len) ? ep.discount[ep_t] : 0.0;
                ep_ret = ep_ret + disc * reward; ep_t += 1;
                if (info == CROWDSIM_INFO_DANGER) { ep_tc += 1; ep_mds += dmin; if constexpr (!MULTI) { ep.ep_too_close[e] = ep_tc; ep.ep_min_dist_sum[e] = ep_mds; } }
                if constexpr (MULTI) dirty_ep = true; else { ep.ep_return[e] = ep_ret; ep.ep_steps[e] = ep_t; }
                if (done) {
                    if (ep_c >= 0) {
                        ep.res_info[ep_c] = (uint8_t)info; ep.res_steps[ep_c] = ep_t;
                        ep.res_time[ep_c] = (info == CROWDSIM_INFO_TIMEOUT) ? k.time_limit : gtime;
                        ep.res_return[ep_c] = ep_ret; ep.res_too_close[ep_c] = ep_tc; ep.res_min_dist_sum[ep_c] = ep_mds;
                        if (ep.res_final_rpos) st2(ep.res_final_rpos, ep_c, pos);
                    }
                    if (A.st.active && !A.has_ar) { A.st.active[e] = 0; act_flag = 0; }
                }
            }
        }
        if (A.has_ar) {
            // consumer side of the auto-reset protocol (include/crowdsim_b200.h): an env that just finished, or is parked
            // waiting, looks at its next-scene slot; a slot the generator publishes later is picked up by a later step
            const bool finished = live && done, parked = !live && want_flag != 0;
            if (finished || parked) {
                const uint8_t sst = MULTI ? ld_relaxed_u8(A.ar.n_state + e) : slot_state;
                if (sst == CROWDSIM_SLOT_READY) install = 1;
                else {
                    act_flag = 0; A.st.active[e] = 0;                             // park: nothing to install (yet)
                    want_flag = (sst == CROWDSIM_SLOT_EXHAUSTED) ? 0 : 1; A.ar.want[e] = want_flag;
                }
            }
        }
    }
    if (A.has_ar) {                                          // warp-uniform
        install = __shfl_sync(CS_FULL, install, rl) && env_ok;
        if constexpr (!MULTI) {
            // single step: the scene goes straight from the slot to the live state (ar_install_*: acquire on the slot flag, copy)
            if (install) {
                if (is_robot) ar_install_robot(A, e);
                else {
                    ar_install_human(A, e, N, a);
                    if (A.io.obs32) { const double2 np_ = ld2_cg(A.ar.n_h_pos, hi); reinterpret_cast<float4 *>(A.io.obs32)[hi] = make_float4((float)np_.x, (float)np_.y, 0.f, 0.f); }
                }
            }
        } else if (install) {
            // acquire on the slot flag (every lane that reads slot data), then the scene (agent.py:47-58 set(px,py,gx,gy,0,0,..))
            (void)ld_acquire_u8(A.ar.n_state + e);
            if (!is_robot) {
                pos = ld2_cg(A.ar.n_h_pos, hi); vel = make_double2(0, 0); goal = ld2_cg(A.ar.n_h_goal, hi); attr = ld2_cg(A.ar.n_h_attr, hi);
            } else {                                         // crowd_sim.py:262,274 + fresh episode accumulators
                pos = make_double2(0.0, -A.ar.circle_radius); goal = make_double2(0.0, A.ar.circle_radius);
                vel = make_double2(0, 0); attr = make_double2(A.ar.robot_radius, A.ar.robot_v_pref);
                theta = CS_PI / 2; gtime = 0.0;
                if (!ROT && A.st.r_theta) A.st.r_theta[e] = CS_PI / 2;
                if (A.has_ep) { ep_t = 0; ep_ret = 0.0; ep_tc = 0; ep_mds = 0.0; ep_c = __ldcg(A.ar.n_case + e); dirty_ep = true; new_case = true; }
                act_flag = 1; A.st.active[e] = 1; want_flag = 0; A.ar.want[e] = 0;
            }
            dirty_kin = true; dirty_scene = true;
        }
        __syncwarp();
        if (install && is_robot) st_release_u8(A.ar.n_state + e, CROWDSIM_SLOT_EMPTY);     // slot data consumed by all lanes of the env
        if (MULTI) act_flag = (uint8_t)__shfl_sync(CS_FULL, (int)act_flag, rl);           // human lanes follow their robot lane's flag
    } else if (MULTI) {
        act_flag = (uint8_t)__shfl_sync(CS_FULL, (int)act_flag, rl);
    }
    if (live && !is_robot && !install) {
        // agent.py:122-135 holonomic step with the ORCA action (float32 values widened) or the Linear action (float64)
        double hx = (double)nv.x, hy = (double)nv.y;
        if constexpr (HLIN) { const double2 lv = linear_human_velocity(pos, goal, attr.y); hx = lv.x; hy = lv.y; }
        pos = make_double2(pos.x + hx * dt, pos.y + hy * dt); vel = make_double2(hx, hy);
        if constexpr (MULTI) dirty_kin = true;
        else {
            st2(A.st.h_pos, hi, pos); st2(A.st.h_vel, hi, vel);
            if (A.io.obs32) reinterpret_cast<float4 *>(A.io.obs32)[hi] = make_float4((float)pos.x, (float)pos.y, HLIN ? (float)hx : nv.x, HLIN ? (float)hy : nv.y);
        }
    }
    }   // step loop

    // ---- multi-step launches: one store of everything the launch changed ----
    if constexpr (MULTI) if (env_ok) {
        if (!is_robot) {
            if (dirty_kin) {
                st2(A.st.h_pos, hi, pos); st2(A.st.h_vel, hi, vel);
                if (A.io.obs32) reinterpret_cast<float4 *>(A.io.obs32)[hi] = make_float4((float)pos.x, (float)pos.y, (float)vel.x, (float)vel.y);
            }
            if (dirty_scene) { st2(A.st.h_goal, hi, goal); st2(A.st.h_attr, hi, attr); }
        } else {
            if (dirty_kin) { st2(A.st.r_pos, e, pos); st2(A.st.r_vel, e, vel); A.st.g_time[e] = gtime; if (ROT) A.st.r_theta[e] = theta; }
            if (dirty_scene) { st2(A.st.r_goal, e, goal); st2(A.st.r_attr, e, attr); }
            if (any_live) {                                  // outputs of the env's last live step
                if (A.io.action_out) st2(A.io.action_out, e, o_act);
                A.io.reward[e] = o_reward; A.io.dmin[e] = o_dmin; A.io.done[e] = (uint8_t)o_done; A.io.info[e] = (uint8_t)o_info;
            }
            if (A.has_ep && dirty_ep) {
                A.ep.ep_steps[e] = ep_t; A.ep.ep_return[e] = ep_ret; A.ep.ep_too_close[e] = ep_tc; A.ep.ep_min_dist_sum[e] = ep_mds;
                if (new_case) A.ep.ep_case[e] = ep_c;
            }
        }
    }
}

}  // namespace cs
