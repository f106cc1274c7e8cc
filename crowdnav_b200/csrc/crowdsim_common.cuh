// crowdsim_common.cuh -- shared pieces of the sm_100a CrowdSim kernels (float64 env arithmetic, staging layout,
// the per-agent ORCA solve on top of orca_device.cuh, launch bookkeeping).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/crowdsim_b200.h"
#include "orca_device.cuh"

namespace cs {

// Kernels launched by this library since load (host-side counter; the bench's gpu_launches claim).
extern unsigned long long g_launches;

#define CS_PI 3.141592653589793

// np.linalg.norm((a, b)): BLAS ddot accumulates a*a, then fma(b, b, .) (see oracle/crowdsim_oracle.c header).
__device__ __forceinline__ double norm2(double a, double b) { return sqrt(fma(b, b, a * a)); }

// crowd_sim/envs/utils/utils.py:4-26 with (x3, y3) = (0, 0)
__device__ __forceinline__ double point_to_segment_dist0(double x1, double y1, double x2, double y2)
{
    const double px = x2 - x1, py = y2 - y1;
    if (px == 0 && py == 0) return norm2(0 - x1, 0 - y1);
    double u = ((0 - x1) * px + (0 - y1) * py) / (px * px + py * py);
    if (u > 1) u = 1; else if (u < 0) u = 0;
    const double x = x1 + u * px, y = y1 + u * py;
    return norm2(x, y);
}

// Linear.predict (crowd_sim/envs/policy/linear.py:15-22): straight to the goal at v_pref, float64 like numpy. An agent standing
// on its goal gets atan2(0, 0) = 0, i.e. it steps +x, as the reference's does.
__device__ __forceinline__ double2 linear_velocity(double2 pos, double2 goal, double v_pref)
{
    const double th = atan2(goal.y - pos.y, goal.x - pos.x);
    return make_double2(cos(th) * v_pref, sin(th) * v_pref);
}
// The same for a human slot; the PARKED slots of rule `mixed` (include/crowdsim_b200.h) never move.
__device__ __forceinline__ double2 linear_human_velocity(double2 pos, double2 goal, double v_pref)
{
    if (pos.x >= CROWDSIM_PARKED_X / 2) return make_double2(0, 0);
    return linear_velocity(pos, goal, v_pref);
}

// Policy selection of the step / lookahead kernels: a compile-time bit set (template parameter LIN), so that the ORCA-human
// instantiations carry no code of the linear ones.
constexpr int kLinHumans = 1;   // human_policy == CROWDSIM_HUMANS_LINEAR
constexpr int kLinRobot = 2;    // robot_policy == CROWDSIM_ROBOT_LINEAR

// Host-side validation of the policy fields of crowdsim_params.
inline bool policies_supported(const crowdsim_params *p)
{
    return p->robot_policy >= CROWDSIM_ROBOT_EXTERNAL_XY && p->robot_policy <= CROWDSIM_ROBOT_LINEAR &&
           (p->human_policy == CROWDSIM_HUMANS_ORCA || p->human_policy == CROWDSIM_HUMANS_LINEAR);
}
inline int lin_bits(const crowdsim_params *p)
{
    return (p->human_policy == CROWDSIM_HUMANS_LINEAR ? kLinHumans : 0) | (p->robot_policy == CROWDSIM_ROBOT_LINEAR ? kLinRobot : 0);
}

__device__ __forceinline__ double2 ld2(const double *p, size_t i) { return reinterpret_cast<const double2 *>(p)[i]; }
__device__ __forceinline__ void st2(double *p, size_t i, double2 v) { reinterpret_cast<double2 *>(p)[i] = v; }
__device__ __forceinline__ double2 ld2_cg(const double *p, size_t i) { return __ldcg(reinterpret_cast<const double2 *>(p) + i); }

// Slot flags of the auto-reset protocol (include/crowdsim_b200.h: crowdsim_autoreset). The generator and the step kernels may
// run concurrently on different streams, so the hand-over is a formal release / acquire pair at gpu scope:
//   generator:  ld.acquire(flag) == EMPTY  ->  write the scene  ->  st.release(flag, READY)
//   consumer:   ld.relaxed(flag) == READY decides; every lane that reads slot data does ld.acquire(flag) first;
//               after the lanes re-converged, st.release(flag, EMPTY)
__device__ __forceinline__ uint8_t ld_relaxed_u8(const uint8_t *p) { unsigned v; asm volatile("ld.relaxed.gpu.global.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return (uint8_t)v; }
__device__ __forceinline__ uint8_t ld_acquire_u8(const uint8_t *p) { unsigned v; asm volatile("ld.acquire.gpu.global.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return (uint8_t)v; }
__device__ __forceinline__ void st_release_u8(uint8_t *p, uint8_t v) { asm volatile("st.release.gpu.global.u8 [%0], %1;" :: "l"(p), "r"((unsigned)v) : "memory"); }

// Device-side copy of the scalar parameters (passed by value as a kernel argument).
struct KParams {
    double time_step, time_limit, success_reward, collision_penalty, discomfort_dist, discomfort_penalty_factor;
    double human_safety_space, robot_safety_space;
    float neighbor_dist, inv_time_horizon, inv_time_step, time_step_f;
    int max_neighbors;   // semantic cap: min(orca max_neighbors, N) -- identical behaviour, a solve never sees more than N candidates
    int nb_alloc;        // shared-memory columns per thread (>= 1)
    int robot_visible, robot_policy;
};

inline KParams make_kparams(const crowdsim_params *p, int N)
{
    KParams k;
    k.time_step = p->time_step; k.time_limit = p->time_limit; k.success_reward = p->success_reward;
    k.collision_penalty = p->collision_penalty; k.discomfort_dist = p->discomfort_dist;
    k.discomfort_penalty_factor = p->discomfort_penalty_factor;
    k.human_safety_space = p->human_safety_space; k.robot_safety_space = p->robot_safety_space;
    k.neighbor_dist = (float)p->neighbor_dist;
    k.inv_time_horizon = 1.0f / (float)p->time_horizon;      // Agent.cpp: invTimeHorizon = 1.0f / timeHorizon_
    k.inv_time_step = 1.0f / (float)p->time_step;            // invTimeStep = 1.0f / sim_->timeStep_
    k.time_step_f = (float)p->time_step;                     // sim_->timeStep_ (Agent::update)
    k.max_neighbors = p->max_neighbors < N ? p->max_neighbors : N; if (k.max_neighbors < 0) k.max_neighbors = 0;
    k.nb_alloc = k.max_neighbors < 1 ? 1 : k.max_neighbors;
    k.robot_visible = p->robot_visible; k.robot_policy = p->robot_policy;
    return k;
}

// Shared-memory staging of one block's environments: L = N + 1 agents per env (humans 0..N-1, robot N).
struct Stage {
    double2 *pos64, *vel64;      // [EPB * L]
    double *rad64;               // [EPB * L]
    float2 *pos32, *vel32;       // [EPB * L]  float32 casts consumed by the ORCA solver
    float *radh, *radr;          // [EPB * L]  (float)(radius + 0.01 + safety) as seen by humans / by the robot
    double2 *act;                // [EPB]      robot velocity applied this step
    double *closest;             // [EPB * L]  per-human clearance of the swept segment test
    float *lines, *proj;         // [4 * maxnb * T] each: per-thread columns (orca::Lines)
};

__host__ __device__ inline size_t stage_bytes(int epb, int L, int maxnb, int threads)
{
    size_t agents = (size_t)epb * L;
    size_t b = agents * (16 + 16 + 8 + 8 + 8 + 4 + 4 + 8) + (size_t)epb * 16;
    b = (b + 15) & ~(size_t)15;
    b += (size_t)2 * 4 * maxnb * threads * sizeof(float);
    return b;
}

// Same staging + the crowd kernel's linearProgram3 queue (step_mid.cuh: mid_lp3_floats(), independent of the block size)
// instead of the generic kernel's 2 x 4 x max_neighbors line / projected-line columns per thread.
__host__ __device__ inline size_t stage_bytes_mid(int epb, int L, int lp3_floats)
{
    size_t agents = (size_t)epb * L;
    size_t b = agents * (16 + 16 + 8 + 8 + 8 + 4 + 4 + 8) + (size_t)epb * 16;
    b = (b + 15) & ~(size_t)15;
    b += (size_t)lp3_floats * sizeof(float);
    return b;
}

__device__ __forceinline__ Stage carve_stage(unsigned char *smem, int epb, int L, int maxnb, int threads)
{
    Stage s; const size_t agents = (size_t)epb * L;
    unsigned char *p = smem;
    s.pos64 = reinterpret_cast<double2 *>(p); p += agents * 16;
    s.vel64 = reinterpret_cast<double2 *>(p); p += agents * 16;
    s.act = reinterpret_cast<double2 *>(p); p += (size_t)epb * 16;
    s.rad64 = reinterpret_cast<double *>(p); p += agents * 8;
    s.closest = reinterpret_cast<double *>(p); p += agents * 8;
    s.pos32 = reinterpret_cast<float2 *>(p); p += agents * 8;
    s.vel32 = reinterpret_cast<float2 *>(p); p += agents * 8;
    s.radh = reinterpret_cast<float *>(p); p += agents * 4;
    s.radr = reinterpret_cast<float *>(p); p += agents * 4;
    p = smem + (((size_t)(p - smem) + 15) & ~(size_t)15);
    s.lines = reinterpret_cast<float *>(p); p += (size_t)4 * maxnb * threads * sizeof(float);
    s.proj = reinterpret_cast<float *>(p);
    return s;
}

// Stage one agent (called by its own lane).
__device__ __forceinline__ void stage_agent(const Stage &s, const KParams &k, int slot, double2 pos, double2 vel, double radius)
{
    s.pos64[slot] = pos; s.vel64[slot] = vel; s.rad64[slot] = radius;
    s.pos32[slot] = make_float2((float)pos.x, (float)pos.y);
    s.vel32[slot] = make_float2((float)vel.x, (float)vel.y);
    s.radh[slot] = (float)(radius + 0.01 + k.human_safety_space);    // orca.py:100-104
    s.radr[slot] = (float)(radius + 0.01 + k.robot_safety_space);
}

// ORCA.predict for agent `a` of local env `le` (a == N: the robot). crowd_sim/envs/policy/orca.py:82-132.
// Candidate order = reference observation order: other humans in env order, robot last iff visible
// (crowd_sim.py:324-327); the robot observes all humans (explorer.py:42).
// linearProgram3 runs in place here: a block-compacted pass with parallel sub-problems (as in step_flat.cuh) was measured
// for this kernel and is neutral at 4096 envs and 3-12 % slower at 65 k envs (N = 10, 20), so it was not kept.
__device__ __forceinline__ orca::V2 orca_predict(const Stage &s, const KParams &k, int le, int a, int N, int L,
                                                 double2 pos, double2 goal, double v_pref, int tid, int threads)
{
    using namespace orca;
    const bool is_robot = (a == N);
    const int base = le * L;
    // orca.py:113-115 preferred velocity in float64 (numpy), then the float32 cast of the rvo2 boundary
    const double gvx = goal.x - pos.x, gvy = goal.y - pos.y;
    const double speed = norm2(gvx, gvy);
    const double pvx = (speed > 1) ? gvx / speed : gvx, pvy = (speed > 1) ? gvy / speed : gvy;
    const V2 pref = mk((float)pvx, (float)pvy);
    const float2 p2 = s.pos32[base + a], v2 = s.vel32[base + a];
    const V2 p = mk(p2.x, p2.y), v = mk(v2.x, v2.y);
    const float *rad_view = is_robot ? s.radr : s.radh;
    const float r = rad_view[base + a];
    const float max_speed = (float)v_pref;

    int cnt = 0;
    const int ncand = (is_robot || !k.robot_visible) ? N : L;
    const Lines Lr = { s.lines + tid, threads };
    const float range_sq0 = sqr(k.neighbor_dist);
    if (k.max_neighbors > 0 && ncand <= 4 * k.nb_alloc) {
        // Neighbour selection by repeated arg-min over cached distances: round n picks the nearest not-yet-taken
        // candidate (ties: lowest scan index, = RVO2's stable insertion order) and builds ORCA line n directly.
        // Uniform control flow; the data-dependent shifting of insert_neighbor was 19 % of the N = 20 kernel's
        // instructions at 11.7 / 32 active lanes (profiles/r01_step_generic_n20_ncu_full.txt); measured gain -13 % at N = 20.
        float *dd = s.proj + tid;                            // distance cache: candidate slot c -> dd[c * threads]
        for (int j = 0; j < ncand; ++j) {
            const float2 q = s.pos32[base + j];
            const float d = abssq(p - mk(q.x, q.y));
            dd[j * threads] = (j != a && d < range_sq0) ? d : __int_as_float(0x7f800000);   // +inf = not a candidate
        }
        unsigned long long taken = 0ull;
        for (int n = 0; n < k.max_neighbors; ++n) {
            float best = __int_as_float(0x7f800000); int bj = -1;
            for (int j = 0; j < ncand; ++j) {
                const float d = dd[j * threads];
                if (d < best && !((taken >> j) & 1ull)) { best = d; bj = j; }
            }
            if (bj < 0) break;
            taken |= 1ull << bj;
            const float2 q = s.pos32[base + bj], w = s.vel32[base + bj];
            V2 lp, ld;
            make_line(p, v, r, mk(q.x, q.y), mk(w.x, w.y), rad_view[base + bj], k.inv_time_horizon, k.inv_time_step, lp, ld);
            Lr.set(cnt++, lp, ld);
        }
    } else if (k.max_neighbors > 0) {
        // RVO2's insertion sort literally (A.2); neighbour list columns live in the (not yet used) proj region
        float *nd = s.proj + tid; int *ni = reinterpret_cast<int *>(s.proj + (size_t)k.nb_alloc * threads) + tid;
        float range_sq = range_sq0;
        for (int j = 0; j < ncand; ++j) {
            if (j == a) continue;
            const float2 q = s.pos32[base + j];
            insert_neighbor(abssq(p - mk(q.x, q.y)), j, nd, ni, threads, cnt, k.max_neighbors, range_sq);
        }
        for (int n = 0; n < cnt; ++n) {
            const int j = ni[n * threads];
            const float2 q = s.pos32[base + j], w = s.vel32[base + j];
            V2 lp, ld;
            make_line(p, v, r, mk(q.x, q.y), mk(w.x, w.y), rad_view[base + j], k.inv_time_horizon, k.inv_time_step, lp, ld);
            Lr.set(n, lp, ld);
        }
    }
    V2 nv;
    const int fail = lp2(Lr, cnt, max_speed, pref, false, nv);
    if (fail < cnt) { const Lines Pr = { s.proj + tid, threads }; lp3(Lr, cnt, fail, max_speed, Pr, nv); }
    return nv;
}

// Envs per block for ~128-thread blocks of L = N + 1 lanes per env.
inline int envs_per_block(int L, int target_threads) { int e = target_threads / L; return e < 1 ? 1 : e; }

}  // namespace cs
