// times_kernel.cu -- CrowdSim.get_human_times (crowd_sim/envs/crowd_sim.py:209-249): after an episode in which the robot
// reached its goal, ONE centralised rvo2 simulation holding the robot (agent 0) and the N humans (agents 1..N) is stepped
// until every human has reached its goal; human_times[i] = global_time of the first step after which human i is within
// its radius of its goal. What the reference does per iteration, and what is reproduced here (sm_100a):
//   * preferred velocity of every agent from the PYTHON-side position (float64 at first, afterwards the simulator's float32
//     position widened: crowd_sim.py:243-245 writes it back), goal - position, normalised if longer than 1 (numpy float64),
//     cast to float32 at the rvo2 boundary;
//   * rvo2 doStep: every agent solves from the same pre-state -- neighbours = all other agents in index order, at most 10
//     within 10 m (Appendix A.2), radius = the agent's plain radius (no + 0.01 here: crowd_sim.py:222-225), maxSpeed =
//     v_pref; then velocity = new velocity, position += velocity * dt IN FLOAT32 (Agent::update);
//   * global_time += dt (float64); the goal test (agent.py:137-138, float64) on the Python-side positions, which at that
//     point still are those of the PREVIOUS iteration (crowd_sim.py:238-245 tests first, copies the positions back after).
// One block per env, one thread per agent; the float32 simulator state lives in shared memory. The solver is the generic
// sequential code of orca_device.cuh (this path runs once per visualised episode; it is not a throughput path).
#include "crowdsim_common.cuh"
#include "orca_spec.cuh"

namespace cs {

struct TimesArgs {
    KParams k;
    int B, N, L, max_steps;
    crowdsim_state st;
    double *human_times;   // [B][N] in/out
    double *g_time_out;    // [B]
    double *final_pos;     // [B][L][2] or NULL, simulator order: robot first
};

__global__ void __launch_bounds__(64) human_times_kernel(const __grid_constant__ TimesArgs A)
{
    using namespace orca;
    extern __shared__ __align__(16) unsigned char smem[];
    const int L = A.L, N = A.N, a = threadIdx.x, e = blockIdx.x;     // a: simulator index, 0 = robot, 1..N = humans
    float2 *s_pos = reinterpret_cast<float2 *>(smem);                // [L] simulator positions / velocities / radii
    float2 *s_vel = s_pos + L;
    float *s_rad = reinterpret_cast<float *>(s_vel + L);
    float *s_cols = s_rad + ((L + 3) & ~3);                           // per-thread columns: 4 x 10 lines + 4 x 10 projected lines
    __shared__ int s_pending;
    const KParams &k = A.k;
    constexpr int M = CROWDSIM_MAX_NEIGHBORS;

    double2 pos, goal, attr, vel0;
    if (a == 0) { pos = ld2(A.st.r_pos, e); goal = ld2(A.st.r_goal, e); attr = ld2(A.st.r_attr, e); vel0 = ld2(A.st.r_vel, e); }
    else { const size_t i = (size_t)e * N + (a - 1); pos = ld2(A.st.h_pos, i); goal = ld2(A.st.h_goal, i); attr = ld2(A.st.h_attr, i); vel0 = ld2(A.st.h_vel, i); }
    double ht = (a > 0) ? A.human_times[(size_t)e * N + (a - 1)] : 1.0;
    double gtime = A.st.g_time[e];
    V2 p = mk((float)pos.x, (float)pos.y), v = mk((float)vel0.x, (float)vel0.y);
    const float r = (float)attr.x, max_speed = (float)attr.y;
    const Lines Lr = { s_cols + a, L }, Pr = { s_cols + (size_t)4 * M * L + a, L };
    const float inf = __int_as_float(0x7f800000);

    for (int it = 0; it < A.max_steps; ++it) {
        if (a == 0) s_pending = 0;
        s_pos[a] = make_float2(p.x, p.y); s_vel[a] = make_float2(v.x, v.y); s_rad[a] = r;
        __syncthreads();
        if (a > 0 && ht == 0.0) atomicOr(&s_pending, 1);             // crowd_sim.py:231 while not all(self.human_times)
        __syncthreads();
        if (!s_pending) break;
        // preferred velocity (crowd_sim.py:229-233)
        const double gvx = goal.x - pos.x, gvy = goal.y - pos.y;
        const double speed = norm2(gvx, gvy);
        const V2 pref = mk((float)((speed > 1) ? gvx / speed : gvx), (float)((speed > 1) ? gvy / speed : gvy));
        // neighbours: all other agents in index order, the <= 10 nearest within range
        float td[M]; int tj[M];
        #pragma unroll
        for (int kk = 0; kk < M; ++kk) { td[kk] = inf; tj[kk] = 0; }
        int cnt = 0;
        if (k.max_neighbors > 0)
            for (int j = 0; j < L; ++j) {
                const float2 q = s_pos[j];
                const float d = abssq(p - mk(q.x, q.y));
                const bool in = (j != a) && d < sqr(k.neighbor_dist);
                cnt += in ? 1 : 0;
                insert_sorted<M>(in ? d : inf, j, td, tj);
            }
        int nl = cnt < k.max_neighbors ? cnt : k.max_neighbors; nl = nl < M ? nl : M;
        #pragma unroll
        for (int kk = 0; kk < M; ++kk)
            if (kk < nl) {
                const int j = tj[kk];
                const float2 q = s_pos[j], w = s_vel[j];
                V2 lp, ld;
                make_line(p, v, r, mk(q.x, q.y), mk(w.x, w.y), s_rad[j], k.inv_time_horizon, k.inv_time_step, lp, ld);
                Lr.set(kk, lp, ld);
            }
        V2 nv;
        const int fail = lp2(Lr, nl, max_speed, pref, false, nv);
        if (fail < nl) lp3(Lr, nl, fail, max_speed, Pr, nv);
        __syncthreads();                                             // every agent solved from the same pre-state
        // Agent::update in float32, then the Python-side mirrors
        v = nv;
        p = p + mk(v.x * k.time_step_f, v.y * k.time_step_f);
        gtime += k.time_step;
        // crowd_sim.py:238-240 runs BEFORE the positions are copied back from the simulator (:243-245): the goal test of this
        // iteration sees the Python-side position of the previous one
        if (a > 0 && ht == 0.0 && norm2(pos.x - goal.x, pos.y - goal.y) < attr.x) ht = gtime;
        pos = make_double2((double)p.x, (double)p.y);
    }
    if (a > 0) A.human_times[(size_t)e * N + (a - 1)] = ht;
    if (a == 0) A.g_time_out[e] = gtime;
    if (A.final_pos) st2(A.final_pos, (size_t)e * L + a, pos);
}

}  // namespace cs

extern "C" int crowdsim_human_times(const crowdsim_params *prm, int B, int N, const crowdsim_state *st, double *human_times,
                                    double *g_time_out, double *final_pos, int max_steps, void *stream)
{
    if (!prm || !st || !human_times || !g_time_out || B < 0 || N < 1 || max_steps < 0) return CROWDSIM_EINVAL;
    if (N > CROWDSIM_MAX_HUMANS || prm->max_neighbors > CROWDSIM_MAX_NEIGHBORS || !cs::policies_supported(prm)) return CROWDSIM_EUNSUPPORTED;
    if (!st->h_pos || !st->h_vel || !st->h_goal || !st->h_attr || !st->r_pos || !st->r_vel || !st->r_goal || !st->r_attr || !st->g_time) return CROWDSIM_EINVAL;
    if (B == 0) return CROWDSIM_OK;
    cs::TimesArgs A;
    A.k = cs::make_kparams(prm, N + 1);                          // a solve sees up to N other agents
    A.B = B; A.N = N; A.L = N + 1; A.max_steps = max_steps; A.st = *st;
    A.human_times = human_times; A.g_time_out = g_time_out; A.final_pos = final_pos;
    const int L = N + 1;
    const size_t smem = (size_t)L * 16 + (size_t)((L + 3) & ~3) * 4 + (size_t)8 * CROWDSIM_MAX_NEIGHBORS * L * 4;
    cs::human_times_kernel<<<B, L, smem, (cudaStream_t)stream>>>(A);
    ++cs::g_launches;
    return (int)cudaGetLastError();
}
