/*
 * include/crowdsim_b200.h -- C ABI of libcrowdsim_b200.so (the drop-in boundary).
 *
 * Batched CrowdSim-v0 physics on one B200: B independent environments, N humans each,
 * stepped in lockstep by hand-written sm_100a kernels. Plain pointers and sizes only; every
 * pointer is a DEVICE pointer owned by the caller (torch, cudaMalloc, ...), no hidden
 * allocation, no synchronisation: calls enqueue work on `stream` (a cudaStream_t passed as
 * void*, NULL = legacy default stream) and return 0, a negative CROWDSIM_E* code for a bad
 * argument, or a positive cudaError_t.
 *
 * What each entry point replaces in the reference (paths relative to /root/reference):
 *   crowdsim_step            crowd_sim/envs/crowd_sim.py:317-420 (CrowdSim.step, update=True) including the
 *                            N x Human.act -> ORCA.predict -> rvo2 doStep (crowd_sim/envs/policy/orca.py:82-132) or
 *                            Linear.predict (crowd_sim/envs/policy/linear.py:15-22, human_policy),
 *                            optionally the robot's own ORCA.predict / Linear.predict (crowd_nav/utils/explorer.py:42), the
 *                            per-step part of Explorer.run_k_episodes (explorer.py:41-72)
 *   crowdsim_step_n          the inner loop of Explorer.run_k_episodes for a robot that decides on device
 *                            (crowd_nav/utils/explorer.py:41-43: robot.act -> env.step, n times), closed on the GPU
 *   crowdsim_orca_act        crowd_sim/envs/utils/robot.py:9-14 with policy ORCA (orca.py:82-132), batched
 *   crowdsim_reset           crowd_sim/envs/crowd_sim.py:251-312 + generators :155-207 (np.random MT19937)
 *   crowdsim_prefetch_scenes the same generators, run ahead of time for the NEXT episode of each env slot
 *                            (explorer.py:35-36: reset() of the following episode)
 *   crowdsim_lookahead_pack  crowd_nav/policy/multi_human_rl.py:35-45 = 81 x env.onestep_lookahead
 *                            (crowd_sim.py:314-315,414-416) + CADRL.propagate (cadrl.py:104-129) +
 *                            CADRL.rotate (cadrl.py:187-222), fused
 *   crowdsim_pack_joint      crowd_sim/envs/utils/state.py:17-18,36-37 (14-tuple) + cadrl.py:187-222 (rotate)
 *   crowdsim_lookahead_humans  the observation of env.onestep_lookahead (crowd_sim.py:314-315,414-416; agent.py:63-74)
 *   crowdsim_occupancy_maps  crowd_nav/policy/multi_human_rl.py:109-163 (MultiHumanRL.build_occupancy_maps)
 *   crowdsim_onestep_lookahead  crowd_sim/envs/crowd_sim.py:314-315 (step(action, update=False)), one action per env
 *   crowdsim_human_times     crowd_sim/envs/crowd_sim.py:209-249 (CrowdSim.get_human_times: the centralised multi-step sim)
 *
 * Layout in HBM (structure of arrays, float64 like the reference's Python floats):
 *   two-vectors are interleaved (x,y) pairs so one agent's pair is one 16-byte load;
 *   human arrays are [B][N][2] (env-major), robot arrays [B][2], scalars [B].
 */
#ifndef CROWDSIM_B200_H
#define CROWDSIM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CROWDSIM_ABI_VERSION 5

/* error codes */
#define CROWDSIM_OK            0
#define CROWDSIM_EINVAL       (-1)   /* NULL required pointer / B,N out of range */
#define CROWDSIM_EUNSUPPORTED (-2)   /* N > CROWDSIM_MAX_HUMANS, max_neighbors > CROWDSIM_MAX_NEIGHBORS, unknown policy, ... */
#define CROWDSIM_ENODEVICE    (-3)   /* no CUDA device / wrong architecture */

#define CROWDSIM_MAX_HUMANS     63   /* N + 1 (robot) agents of one env are staged together in shared memory */
#define CROWDSIM_MAX_NEIGHBORS  10   /* orca.py:62 hard-codes max_neighbors = 10 */

/* info codes: crowd_sim/envs/utils/info.py:1-38 */
#define CROWDSIM_INFO_NOTHING   0
#define CROWDSIM_INFO_DANGER    1
#define CROWDSIM_INFO_REACHGOAL 2
#define CROWDSIM_INFO_COLLISION 3
#define CROWDSIM_INFO_TIMEOUT   4

/* robot_policy */
#define CROWDSIM_ROBOT_EXTERNAL_XY  0  /* holonomic ActionXY supplied by the caller (CADRL/LSTM-RL/SARL/Linear) */
#define CROWDSIM_ROBOT_ORCA         1  /* robot runs ORCA inside the step kernel (test.py --policy orca) */
#define CROWDSIM_ROBOT_EXTERNAL_ROT 2  /* unicycle ActionRot (v, r) supplied by the caller (agent.py:115-118,133-135) */
#define CROWDSIM_ROBOT_LINEAR       3  /* robot runs Linear inside the step kernel (test.py --policy linear): Linear.predict
                                          (crowd_sim/envs/policy/linear.py:15-22) of its pre-step state, io->action unused */

/* human_policy: env.config [humans] policy, crowd_sim/envs/policy/policy_factory.py:9-12 (crowd_sim.py:317-326 human.act) */
#define CROWDSIM_HUMANS_ORCA   0  /* ORCA.predict (orca.py:82-132) */
#define CROWDSIM_HUMANS_LINEAR 1  /* Linear.predict (linear.py:15-22): theta = atan2(gy - py, gx - px) in float64, velocity
                                     (cos theta * v_pref, sin theta * v_pref); no neighbour scan. A human standing on its goal
                                     steps +x (atan2(0, 0) = 0) like the reference's; PARKED slots of `mixed` stay still. */

/* scenario rules: crowd_sim.py:84-153 */
#define CROWDSIM_RULE_CIRCLE 0
#define CROWDSIM_RULE_SQUARE 1
/* crowd_sim.py:103-151: per scene 0..5 humans, standing (20 %) or two circle- + the rest square-crossing. The arrays keep
 * their fixed N; unused human slots are PARKED at position = goal = (CROWDSIM_PARKED_X + 100 i, CROWDSIM_PARKED_X): out of
 * every neighbour range (neighbor_dist must stay below 100) and of every collision / min-distance test, never moving.
 * A consumer counts the present humans of env e as #{i : h_pos[e][i].x < CROWDSIM_PARKED_X / 2}. */
#define CROWDSIM_RULE_MIXED 2
#define CROWDSIM_PARKED_X 1.0e6

typedef struct crowdsim_params {
    /* crowd_nav/configs/env.config [env] / [reward]; crowd_sim.py:51-60 */
    double time_step;                 /* 0.25 */
    double time_limit;                /* 25   */
    double success_reward;            /* 1    */
    double collision_penalty;         /* -0.25 */
    double discomfort_dist;           /* 0.2  */
    double discomfort_penalty_factor; /* 0.5  */
    /* ORCA constants, hard-coded in orca.py:61-64; cast to float32 at the rvo2 boundary */
    double neighbor_dist;             /* 10 */
    double time_horizon;              /* 5  */
    int32_t max_neighbors;            /* 10 */
    /* orca.py:100-104: radius + 0.01 + safety_space (float64 sum, then cast) */
    double human_safety_space;        /* 0 */
    double robot_safety_space;        /* 0 (train.py:121-127 sets 0.15 for IL with an invisible robot) */
    int32_t robot_visible;            /* env.config [robot] visible; crowd_sim.py:325-327 */
    int32_t robot_policy;             /* CROWDSIM_ROBOT_* */
    int32_t human_policy;             /* CROWDSIM_HUMANS_* (appended last: zero-filled initialisers mean ORCA humans) */
} crowdsim_params;

/* Agent state. Mutable arrays are updated in place by crowdsim_step (agent.py:122-135). */
typedef struct crowdsim_state {
    double *h_pos;    /* [B][N][2] human px,py            (mutable) */
    double *h_vel;    /* [B][N][2] human vx,vy            (mutable) */
    double *h_goal;   /* [B][N][2] human gx,gy                      */
    double *h_attr;   /* [B][N][2] human radius, v_pref             */
    double *r_pos;    /* [B][2]    robot px,py            (mutable) */
    double *r_vel;    /* [B][2]    robot vx,vy            (mutable) */
    double *r_goal;   /* [B][2]    robot gx,gy                      */
    double *r_attr;   /* [B][2]    robot radius, v_pref             */
    double *r_theta;  /* [B]       robot heading          (mutable, unicycle only) */
    double *g_time;   /* [B]       env.global_time        (mutable) */
    uint8_t *active;  /* [B] or NULL: 0 = env frozen (episode over, waiting for reset); NULL = all live */
} crowdsim_state;

/* Per-step inputs / outputs of crowdsim_step. */
typedef struct crowdsim_step_io {
    const double *action; /* [B][2] robot action (vx,vy) or (v,r); ignored (may be NULL) for CROWDSIM_ROBOT_ORCA / _LINEAR */
    double *action_out;   /* [B][2] or NULL: the holonomic velocity actually applied to the robot */
    double *reward;       /* [B] */
    double *dmin;         /* [B] min robot-human clearance this step (inf if N == 0) */
    uint8_t *done;        /* [B] */
    uint8_t *info;        /* [B] CROWDSIM_INFO_* */
    float *obs32;         /* [B][N][4] or NULL: the observation after the step as float32 (px, py, vx, vy) per human -- the
                             cast the value-network policies apply anyway (crowd_nav/policy/multi_human_rl.py:43); velocities
                             are float32-valued ORCA outputs, so only the positions are rounded. For host-side callers: a
                             third of the bytes of the float64 state arrays on the device->host link. */
} crowdsim_step_io;

/*
 * Episode bookkeeping of Explorer.run_k_episodes (explorer.py:35-72), all optional (pass NULL struct pointer
 * to skip). Slot arrays are per env slot; result arrays are indexed by the episode's case slot `ep_case[e]`
 * (0..k-1) and written once when the episode terminates, after which active[e] is cleared (if present).
 */
typedef struct crowdsim_episodes {
    int32_t *ep_case;        /* [B] index into the result arrays, <0 = do not record */
    int32_t *ep_steps;       /* [B] steps taken so far in the running episode */
    double  *ep_return;      /* [B] running sum_t discount[t] * reward_t (explorer.py:71-72) */
    int32_t *ep_too_close;   /* [B] running count of Danger steps (explorer.py:48-49) */
    double  *ep_min_dist_sum;/* [B] running sum of Danger min_dist (explorer.py:50) */
    const double *discount;  /* [discount_len] pow(gamma, t*time_step*v_pref), host-computed with C pow */
    int32_t discount_len;
    /* results, one row per finished episode */
    uint8_t *res_info;       /* [k] terminal CROWDSIM_INFO_* */
    int32_t *res_steps;      /* [k] */
    double  *res_time;       /* [k] global_time after the terminal step (time_limit for timeouts, explorer.py:62) */
    double  *res_return;     /* [k] */
    int32_t *res_too_close;  /* [k] */
    double  *res_min_dist_sum;/*[k] */
    double  *res_final_rpos; /* [k][2] or NULL: robot position after the terminal step (parity evidence) */
} crowdsim_episodes;

/*
 * Auto-reset with prefetched scenes (optional, pass NULL to crowdsim_step to disable).
 * Every env slot owns a "next scene" buffer. crowdsim_prefetch_scenes (any stream, may overlap with steps) fills
 * slots whose n_state is EMPTY and marks them READY; crowdsim_step, when an env's episode terminates, installs the
 * READY scene into the live state in the same launch (fresh episode, global_time 0, velocities 0, accumulators
 * cleared, ep_case = n_case) and marks the slot EMPTY again. If the scene is not ready yet the env is parked
 * (active = 0, want = 1) and installed by a later step; EXHAUSTED slots (case queue empty) just go inactive.
 * Single-writer protocol: only the generator moves EMPTY -> READY/EXHAUSTED, only the step kernel moves READY -> EMPTY;
 * both sides publish with st.release.gpu and read slot data behind ld.acquire.gpu, so the generator may run concurrently
 * with steps of the same batch on another stream.
 * Requires crowdsim_state.active != NULL.
 */
#define CROWDSIM_SLOT_EMPTY     0
#define CROWDSIM_SLOT_READY     1
#define CROWDSIM_SLOT_EXHAUSTED 2
typedef struct crowdsim_autoreset {
    double *n_h_pos;     /* [B][N][2] next scene: human start positions */
    double *n_h_goal;    /* [B][N][2] human goals */
    double *n_h_attr;    /* [B][N][2] human radius, v_pref */
    int32_t *n_case;     /* [B] case index of the prefetched scene (-1 = untracked) */
    uint8_t *n_state;    /* [B] CROWDSIM_SLOT_* */
    uint8_t *want;       /* [B] 1 = env finished and is waiting for a scene */
    double circle_radius;  /* robot start/goal (0, -R) -> (0, R), crowd_sim.py:274 */
    double robot_radius, robot_v_pref;
} crowdsim_autoreset;

/* Scenario generation request for crowdsim_reset / crowdsim_prefetch_scenes. */
typedef struct crowdsim_reset_args {
    const uint8_t *mask;     /* [B] or NULL: reset only envs with mask[e] != 0 (NULL = all) */
    uint32_t *seed;          /* [B] MT19937 seed per env (crowd_sim.py:272-276: offset[phase] + case); after a masked env
                                has been reset its entry is advanced by seed_stride (next scene of that slot) */
    uint32_t seed_stride;    /* 0 = leave seeds untouched */
    int32_t rule;            /* CROWDSIM_RULE_* */
    double circle_radius;    /* env.config [sim] circle_radius = 4 */
    double square_width;     /* env.config [sim] square_width  = 10 */
    double human_radius;     /* env.config [humans] radius = 0.3 */
    double human_v_pref;     /* env.config [humans] v_pref = 1   */
    double robot_radius;     /* env.config [robot] radius = 0.3  */
    double robot_v_pref;     /* env.config [robot] v_pref = 1    */
    double discomfort_dist;  /* 0.2 (min initial separation, crowd_sim.py:168) */
    int32_t randomize_attributes; /* env.config [env] randomize_attributes (agent.py:39-45) */
    /* Optional case work-queue (Explorer.run_k_episodes over k cases with fewer slots): when case_counter != NULL the
     * seed of a generated scene is seed_base + c (see case_wrap below) with c = atomicAdd(case_counter, 1); c >= case_total => no scene
     * (prefetch marks the slot EXHAUSTED). `seed`/`seed_stride` are ignored then. */
    int32_t *case_counter;
    int32_t case_total;
    uint32_t seed_base;
    /* Wrap of the case numbers inside a phase (crowd_sim.py:283: case_counter = (case_counter + 1) % case_size): when
     * case_wrap > 0 the seed of queue entry c is seed_base + (case_first + c) % case_wrap, i.e. seed_base = offset[phase]
     * and the k cases of a run that crosses the end of the phase's case range continue at case 0 like the reference's;
     * case_wrap = 0: seed_base + c. */
    int32_t case_first;
    int32_t case_wrap;
} crowdsim_reset_args;

/* Library / device probing (host only, no kernel launch). */
int crowdsim_abi_version(void);
int crowdsim_device_check(int *sm_count, int *cc_major, int *cc_minor);
/* Kernels launched by this library since load (the bench's gpu_launches claim). */
unsigned long long crowdsim_launch_count(void);
/* Test hook: 1 = use the generic one-thread-per-agent step kernel for every N (default 0: N <= 5 uses the
 * register-resident small-crowd kernel). Both are held to the same bit-exact parity bar. */
void crowdsim_debug_force_generic(int on);

/* Host plumbing for callers that keep several env batches in flight from an interpreter (batched.HostStepper.launch /
 * wait; the reference's loop blocks in env.step, crowd_nav/utils/explorer.py:42-43): replay a captured CUDA graph
 * (cudaGraphExec_t) of one batch's step on `stream` and record `done_event` (cudaEvent_t, may be NULL) behind it / block
 * until that event has completed. No kernel of this library is launched directly by these two calls. */
int crowdsim_graph_launch(void *graph_exec, void *stream, void *done_event);
int crowdsim_event_wait(void *event);
/* The round-robin of a host that keeps n independent env batches in flight, natively: `rounds` times, for every batch i:
 * wait for events[i] (its previous step: results are in its pinned host buffers), memcpy copy_bytes from copy_src[i] to
 * copy_dst[i] (the host-side hand-over between two steps -- e.g. next_action -> action: "apply the decision the device
 * computed"; NULL pointers or copy_bytes = 0: none), replay graph_execs[i] on streams[i] and record events[i] behind it.
 * graph_execs_alt (may be NULL) + alt_period > 1: round number first_round + r replays graph_execs only when it is a multiple
 * of alt_period and graph_execs_alt otherwise (e.g. the step graph with / without the scene-refill branch).
 * On return the last step of every batch is still in flight (wait with crowdsim_event_wait). No kernel of this library is
 * launched directly. batched.HostStepperGroup wraps it. */
int crowdsim_host_pump(int n, void *const *graph_execs, void *const *graph_execs_alt, int alt_period, int first_round,
                       void *const *streams, void *const *events,
                       void *const *copy_dst, const void *const *copy_src, size_t copy_bytes, int rounds);

/* One lockstep env-step for B envs. `ep` and `ar` may be NULL. */
int crowdsim_step(const crowdsim_params *prm, int B, int N, crowdsim_state *st, crowdsim_step_io *io,
                  crowdsim_episodes *ep, const crowdsim_autoreset *ar, void *stream);

/*
 * n_steps lockstep env-steps in one call: exactly n_steps x crowdsim_step(prm, B, N, st, io, ep, ar) -- same final state,
 * same episode rows, same slot hand-overs; `io` holds the outputs of each env's LAST live step. With a robot that decides on
 * device (CROWDSIM_ROBOT_ORCA or CROWDSIM_ROBOT_LINEAR) nothing leaves the device between the steps of the reference's episode loop
 * (crowd_nav/utils/explorer.py:41-43), so for N <= 5 the whole call is ONE kernel launch that keeps every env's state in
 * registers across the steps (one load, n_steps solves, one store); an env whose episode ends installs its prefetched next
 * scene on the spot and goes on (a second termination inside the same call finds the slot EMPTY and parks until the next
 * crowdsim_prefetch_scenes, as n_steps single steps without a refill in between would). Other configurations
 * (external robot actions: the same io->action every step; N > 5) run n_steps launches.
 */
int crowdsim_step_n(const crowdsim_params *prm, int B, int N, crowdsim_state *st, crowdsim_step_io *io,
                    crowdsim_episodes *ep, const crowdsim_autoreset *ar, int n_steps, void *stream);

/* Robot ORCA action from the current state, no mutation: action_out[B][2]. */
int crowdsim_orca_act(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, double *action_out,
                      void *stream);

/* (Re)generate scenarios for the masked envs; also zeroes g_time, velocities, sets theta = pi/2, and,
 * when `ep` is given, clears the slot accumulators. Sets active[e] = 1 if `st->active` is present. */
int crowdsim_reset(const crowdsim_reset_args *args, int B, int N, crowdsim_state *st, crowdsim_episodes *ep,
                   void *stream);

/* Fill the EMPTY next-scene slots of `ar` (generator side of the auto-reset protocol above). `args->mask` is ignored. */
int crowdsim_prefetch_scenes(const crowdsim_reset_args *args, int B, int N, const crowdsim_autoreset *ar, void *stream);

/*
 * Rotated joint state of the CURRENT state for value-net policies: out[B][N][13] float32
 * (cadrl.py:187-222 applied to the 14-tuple of state.py:17-18,36-37 after the float32 cast of
 * multi_human_rl.py:43). kinematics_unicycle selects theta handling (cadrl.py:205-209).
 */
int crowdsim_pack_joint(int B, int N, const crowdsim_state *st, int kinematics_unicycle, float *out, void *stream);

/*
 * One-step lookahead for A candidate robot actions per env (multi_human_rl.py:35-45 with query_env=true):
 * the N human ORCA solves are done once per env and shared by all A actions. Outputs:
 *   out_states [B][A][N][13] float32  rotate(next_self_state + next_human_state)
 *   out_reward [B][A]        float64  reward of step(action, update=False)
 * actions [A][2] float64 are shared by all envs (CADRL.build_action_space, cadrl.py:82-102).
 * Nothing is mutated.
 */
int crowdsim_lookahead_pack(const crowdsim_params *prm, int B, int N, const crowdsim_state *st,
                            const double *actions, int A, int kinematics_unicycle,
                            float *out_states, double *out_reward, void *stream);

/*
 * The humans' next observable states for the current state and the humans' own ORCA decisions -- what
 * env.onestep_lookahead(action) returns as `ob` (it does not depend on the robot's action): next_h_pos, next_h_vel
 * [B][N][2] float64. Nothing is mutated.
 */
int crowdsim_lookahead_humans(const crowdsim_params *prm, int B, int N, const crowdsim_state *st,
                              double *next_h_pos, double *next_h_vel, void *stream);

/*
 * Occupancy maps of MultiHumanRL.build_occupancy_maps (multi_human_rl.py:109-163; policy.config [om] cell_num,
 * cell_size, om_channel_size) for B x N humans given as [B][N][2] float64 position / velocity arrays (the live state or
 * the output of crowdsim_lookahead_humans): out [B][N][cell_num^2 * channels] float32, cell-major, channels 1 (occupied),
 * 2 (mean vx, vy of the occupants in the human's velocity-aligned frame) or 3 (occupied, mean vx, mean vy).
 * N >= 2 (the reference raises for a single human); cell_num^2 <= 64.
 */
int crowdsim_occupancy_maps(int B, int N, const double *h_pos, const double *h_vel, int cell_num, double cell_size,
                            int channels, float *out, void *stream);

/*
 * env.onestep_lookahead(action) = step(action, update=False) (crowd_sim/envs/crowd_sim.py:314-315, 414-416) for one robot
 * action PER ENV: io->reward / dmin / done / info (and action_out) are those step() would return, next_h_pos / next_h_vel
 * [B][N][2] the humans' next observable states (agent.py:63-74); state, time and bookkeeping are NOT modified (the env must be
 * active). For the 81-action sweep of the value-network policies use crowdsim_lookahead_pack.
 */
int crowdsim_onestep_lookahead(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, crowdsim_step_io *io,
                               double *next_h_pos, double *next_h_vel, void *stream);

/*
 * CrowdSim.get_human_times (crowd_sim/envs/crowd_sim.py:209-249): from the CURRENT state (an episode the robot has finished
 * at its goal) one centralised ORCA simulation of the robot and all N humans -- every agent solves from the same pre-state,
 * radius = the plain agent radius, positions advance in float32 like rvo2's own -- is stepped until every human has reached
 * its goal (at most max_steps steps). human_times [B][N] float64 in/out: entries that are already non-zero (humans that
 * arrived during the episode, crowd_sim.py:404-407) are kept, the others receive the global_time of their arrival (0 if
 * max_steps ran out). g_time_out [B]: env.global_time afterwards. final_pos [B][N+1][2] or NULL: the agents' final
 * positions, robot first. The state arrays are NOT modified. N >= 1.
 */
int crowdsim_human_times(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, double *human_times,
                         double *g_time_out, double *final_pos, int max_steps, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CROWDSIM_B200_H */
