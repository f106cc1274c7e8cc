// pack_kernel.cu -- JointState packing and the fused one-step lookahead for value-network robot policies (sm_100a).
//
// crowdsim_pack_joint      current state -> rotate(self_state + human_state) rows, [B][N][13] float32:
//                          crowd_sim/envs/utils/state.py:17-18,36-37 (14-tuple), crowd_nav/policy/multi_human_rl.py:98-107
//                          (transform: float32 cast) and crowd_nav/policy/cadrl.py:187-222 (rotate).
// crowdsim_lookahead_pack  the inner loop of MultiHumanRL.predict / CADRL.predict (multi_human_rl.py:35-45, query_env=true):
//                          for each of A candidate actions, env.onestep_lookahead(action) (crowd_sim.py:314-315,414-416,
//                          agent.py:63-74), CADRL.propagate (cadrl.py:104-129) and rotate. The reference re-solves the N human
//                          ORCA problems for every action although they do not depend on it; here they are solved once
//                          per env (same lane mapping and staging as the step kernel) and shared by the A actions.
//
// Output rows are float32 like the reference's torch tensors; atan2f/cosf/sinf are CUDA's single-precision
// functions (the reference's are torch CPU's), so parity on these rows is a 1e-5 tolerance, not bit-exact.
// Output of one env is A*N*13 contiguous floats: it is assembled in a shared-memory tile and written back with
// fully coalesced stores.
#include <type_traits>
#include "crowdsim_common.cuh"

namespace cs {

// cadrl.py:187-222 on one 14-tuple already cast to float32.
__device__ __forceinline__ void rotate_self(float px, float py, float vx, float vy, float gx, float gy,
                                            float &rot_c, float &rot_s, float &rot, float &dg, float &rvx, float &rvy)
{
    const float dx = gx - px, dy = gy - py;
    rot = atan2f(dy, dx);
    rot_c = cosf(rot); rot_s = sinf(rot);
    dg = sqrtf(dx * dx + dy * dy);
    rvx = vx * rot_c + vy * rot_s;
    rvy = vy * rot_c - vx * rot_s;
}

__device__ __forceinline__ void rotate_row(float *out, float px, float py, float radius, float v_pref, float theta_out,
                                           float dg, float rvx, float rvy, float c, float s,
                                           float hx, float hy, float hvx, float hvy, float hr)
{
    out[0] = dg; out[1] = v_pref; out[2] = theta_out; out[3] = radius; out[4] = rvx; out[5] = rvy;
    out[6] = (hx - px) * c + (hy - py) * s;
    out[7] = (hy - py) * c - (hx - px) * s;
    out[8] = hvx * c + hvy * s;
    out[9] = hvy * c - hvx * s;
    out[10] = hr;
    { const float ax = px - hx, ay = py - hy; out[11] = sqrtf(ax * ax + ay * ay); }
    out[12] = radius + hr;
}

struct PackArgs { int B, N, unicycle; crowdsim_state st; float *out; };

__global__ void __launch_bounds__(128) pack_joint_kernel(const __grid_constant__ PackArgs A)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)A.B * A.N) return;
    const int e = (int)(idx / A.N);
    const double2 rp = ld2(A.st.r_pos, e), rv = ld2(A.st.r_vel, e), rg = ld2(A.st.r_goal, e), ra = ld2(A.st.r_attr, e);
    const double2 hp = ld2(A.st.h_pos, idx), hv = ld2(A.st.h_vel, idx), ha = ld2(A.st.h_attr, idx);
    const float th = (A.unicycle && A.st.r_theta) ? (float)A.st.r_theta[e] : 0.f;
    float c, s, rot, dg, rvx, rvy;
    rotate_self((float)rp.x, (float)rp.y, (float)rv.x, (float)rv.y, (float)rg.x, (float)rg.y, c, s, rot, dg, rvx, rvy);
    float row[13];
    rotate_row(row, (float)rp.x, (float)rp.y, (float)ra.x, (float)ra.y, A.unicycle ? (th - rot) : 0.f, dg, rvx, rvy, c, s,
               (float)hp.x, (float)hp.y, (float)hv.x, (float)hv.y, (float)ha.x);
    float *o = A.out + idx * 13;
    #pragma unroll
    for (int i = 0; i < 13; ++i) o[i] = row[i];
}

struct LookArgs {
    KParams k;
    int B, N, L, EPB, A, unicycle;
    crowdsim_state st;
    const double *actions;
    float *out_states;
    double *out_reward;
};

// HLIN: the humans follow Linear.predict (float64 velocities, kept as such for the next positions) instead of ORCA.
template <bool HLIN = false>
__global__ void __launch_bounds__(256) lookahead_kernel(const __grid_constant__ LookArgs G)
{
    using HVel = typename std::conditional<HLIN, double2, float2>::type;
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = blockDim.x, tid = threadIdx.x;
    const int N = G.N, L = G.L, A = G.A;
    const KParams &k = G.k;
    const Stage s = carve_stage(smem, G.EPB, L, k.nb_alloc, T);
    // extra regions behind the solver staging
    unsigned char *xp = smem + stage_bytes(G.EPB, L, k.nb_alloc, T);
    double2 *s_goal = reinterpret_cast<double2 *>(xp); xp += (size_t)G.EPB * 16;     // robot goal
    double2 *s_rattr = reinterpret_cast<double2 *>(xp); xp += (size_t)G.EPB * 16;    // robot radius, v_pref
    double2 *s_thtime = reinterpret_cast<double2 *>(xp); xp += (size_t)G.EPB * 16;   // robot theta, global_time
    double2 *s_actions = reinterpret_cast<double2 *>(xp); xp += (size_t)A * 16;
    HVel *s_nvel = reinterpret_cast<HVel *>(xp); xp += (size_t)G.EPB * L * sizeof(HVel);  // human actions
    float *tile = reinterpret_cast<float *>(xp);                                      // [A][N][13]

    const int le = tid / L, a = tid - le * L;
    const int e = blockIdx.x * G.EPB + le;
    const bool is_robot = (a == N);
    const bool live = (e < G.B);

    double2 pos = make_double2(0, 0), vel = pos, goal = pos, attr = pos;
    if (live) {
        if (!is_robot) { const size_t i = (size_t)e * N + a; pos = ld2(G.st.h_pos, i); vel = ld2(G.st.h_vel, i); goal = ld2(G.st.h_goal, i); attr = ld2(G.st.h_attr, i); }
        else {
            pos = ld2(G.st.r_pos, e); vel = ld2(G.st.r_vel, e); goal = ld2(G.st.r_goal, e); attr = ld2(G.st.r_attr, e);
            s_goal[le] = goal; s_rattr[le] = attr;
            s_thtime[le] = make_double2((G.st.r_theta ? G.st.r_theta[e] : 0.0), G.st.g_time[e]);
        }
    }
    stage_agent(s, k, tid, pos, vel, attr.x);
    for (int i = tid; i < A; i += T) s_actions[i] = ld2(G.actions, i);
    __syncthreads();

    if (live && !is_robot) {
        if constexpr (HLIN) s_nvel[tid] = linear_human_velocity(pos, goal, attr.y);
        else { const orca::V2 nv = orca_predict(s, k, le, a, N, L, pos, goal, attr.y, tid, T); s_nvel[tid] = make_float2(nv.x, nv.y); }
    }
    __syncthreads();

    const double dt = k.time_step;
    const int row_floats = N * 13;
    for (int l2 = 0; l2 < G.EPB; ++l2) {
        const int e2 = blockIdx.x * G.EPB + l2;
        if (e2 >= G.B) break;                      // uniform across the block
        const int base = l2 * L;
        for (int kk = tid; kk < A; kk += T) {
            const double2 act = s_actions[kk];
            const double2 rp = s.pos64[base + N], rg = s_goal[l2], ra = s_rattr[l2], tt = s_thtime[l2];
            // world-frame robot velocity of this action (crowd_sim.py:336-341)
            double avx = act.x, avy = act.y;
            if (G.unicycle) { avx = act.x * cos(act.y + tt.x); avy = act.x * sin(act.y + tt.x); }
            double dmin = __longlong_as_double(0x7ff0000000000000LL); bool collision = false;
            for (int i = 0; i < N; ++i) {
                const double2 hp = s.pos64[base + i], hv = s.vel64[base + i];
                const double px = hp.x - rp.x, py = hp.y - rp.y;
                const double vx = hv.x - avx, vy = hv.y - avy;
                const double ex = px + vx * dt, ey = py + vy * dt;
                const double c = point_to_segment_dist0(px, py, ex, ey) - s.rad64[base + i] - ra.x;
                if (c < 0) { collision = true; break; } else if (c < dmin) dmin = c;
            }
            // cadrl.py:104-129 propagate(self_state, action); agent.py:110-120 compute_position for the goal test
            double npx, npy, nvx, nvy, nth = tt.x, gpx, gpy;
            if (!G.unicycle) { npx = rp.x + act.x * dt; npy = rp.y + act.y * dt; nvx = act.x; nvy = act.y; gpx = npx; gpy = npy; }
            else {
                nth = tt.x + act.y; nvx = act.x * cos(nth); nvy = act.x * sin(nth);
                npx = rp.x + nvx * dt; npy = rp.y + nvy * dt;
                gpx = rp.x + cos(nth) * act.x * dt; gpy = rp.y + sin(nth) * act.x * dt;
            }
            const bool reaching_goal = norm2(gpx - rg.x, gpy - rg.y) < ra.x;
            double reward;
            if (tt.y >= k.time_limit - 1) reward = 0;
            else if (collision) reward = k.collision_penalty;
            else if (reaching_goal) reward = k.success_reward;
            else if (dmin < k.discomfort_dist) reward = (dmin - k.discomfort_dist) * k.discomfort_penalty_factor * dt;
            else reward = 0;
            G.out_reward[(size_t)e2 * A + kk] = reward;

            float c, sn, rot, dg, rvx, rvy;
            const float fpx = (float)npx, fpy = (float)npy;
            rotate_self(fpx, fpy, (float)nvx, (float)nvy, (float)rg.x, (float)rg.y, c, sn, rot, dg, rvx, rvy);
            const float th_out = G.unicycle ? ((float)nth - rot) : 0.f;
            for (int i = 0; i < N; ++i) {
                const double2 hp = s.pos64[base + i]; const HVel hn = s_nvel[base + i];
                // agent.py:63-74 get_next_observable_state(human_action)
                const double nhx = hp.x + (double)hn.x * dt, nhy = hp.y + (double)hn.y * dt;
                rotate_row(tile + (size_t)kk * row_floats + i * 13, fpx, fpy, (float)ra.x, (float)ra.y, th_out, dg, rvx, rvy, c, sn,
                           (float)nhx, (float)nhy, (float)hn.x, (float)hn.y, (float)s.rad64[base + i]);
            }
        }
        __syncthreads();
        float *dst = G.out_states + (size_t)e2 * A * row_floats;
        const int total = A * row_floats;
        for (int i = tid; i < total; i += T) dst[i] = tile[i];
        __syncthreads();
    }
}


// ---- onestep_lookahead's observation (crowd_sim.py:414-416, agent.py:63-74): the humans' next observable states for the
// CURRENT state, nothing mutated. Same staging and solver as the lookahead kernel. ----
struct NextArgs { KParams k; int B, N, L, EPB; crowdsim_state st; double *next_pos, *next_vel; };

template <bool HLIN = false>
__global__ void __launch_bounds__(256) lookahead_humans_kernel(const __grid_constant__ NextArgs G)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = blockDim.x, tid = threadIdx.x;
    const int N = G.N, L = G.L;
    const KParams &k = G.k;
    const Stage s = carve_stage(smem, G.EPB, L, k.nb_alloc, T);
    const int le = tid / L, a = tid - le * L;
    const int e = blockIdx.x * G.EPB + le;
    const bool is_robot = (a == N);
    const bool live = (e < G.B);
    double2 pos = make_double2(0, 0), vel = pos, goal = pos, attr = pos;
    if (live) {
        if (!is_robot) { const size_t i = (size_t)e * N + a; pos = ld2(G.st.h_pos, i); vel = ld2(G.st.h_vel, i); goal = ld2(G.st.h_goal, i); attr = ld2(G.st.h_attr, i); }
        else { pos = ld2(G.st.r_pos, e); vel = ld2(G.st.r_vel, e); attr = ld2(G.st.r_attr, e); }
    }
    stage_agent(s, k, tid, pos, vel, attr.x);
    __syncthreads();
    if (live && !is_robot) {
        double hx, hy;
        if constexpr (HLIN) { const double2 lv = linear_human_velocity(pos, goal, attr.y); hx = lv.x; hy = lv.y; }
        else { const orca::V2 nv = orca_predict(s, k, le, a, N, L, pos, goal, attr.y, tid, T); hx = (double)nv.x; hy = (double)nv.y; }
        const size_t i = (size_t)e * N + a;
        st2(G.next_pos, i, make_double2(pos.x + hx * k.time_step, pos.y + hy * k.time_step));
        st2(G.next_vel, i, make_double2(hx, hy));
    }
}

// ---- MultiHumanRL.build_occupancy_maps (crowd_nav/policy/multi_human_rl.py:109-163): for every human i a cell_num x
// cell_num grid (cell_size metres per cell) centred on i and aligned with i's velocity; channels = 1: occupancy,
// 2: mean (vx, vy) of the occupants in i's frame, 3: (occupied, mean vx, mean vy). One thread per (env, human);
// float64 like the reference's numpy code, output float32 like its torch tensor. ----
#define CS_OM_MAX_CELLS 64
struct OmArgs { int B, N, cell_num, channels; double cell_size; const double *pos, *vel; float *out; };

__global__ void __launch_bounds__(128) occupancy_kernel(const __grid_constant__ OmArgs G)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)G.B * G.N) return;
    const int N = G.N, e = (int)(idx / N), i = (int)(idx - (size_t)e * N);
    const int cells = G.cell_num * G.cell_num, C = G.channels;
    double sx[CS_OM_MAX_CELLS], sy[CS_OM_MAX_CELLS]; int cnt[CS_OM_MAX_CELLS];
    for (int c = 0; c < cells; ++c) { sx[c] = 0.0; sy[c] = 0.0; cnt[c] = 0; }
    const double2 pi = ld2(G.pos, idx), vi = ld2(G.vel, idx);
    const double angle = atan2(vi.y, vi.x);                                  // :124 new x-axis along the human's velocity
    const double half = (double)G.cell_num / 2;
    for (int j = 0; j < N; ++j) {
        if (j == i) continue;
        const double2 pj = ld2(G.pos, (size_t)e * N + j), vj = ld2(G.vel, (size_t)e * N + j);
        const double ox = pj.x - pi.x, oy = pj.y - pi.y;
        const double rot = atan2(oy, ox) - angle;
        const double dist = sqrt(ox * ox + oy * oy);                         // :127 np.linalg.norm(axis=0)
        const double rx = cos(rot) * dist, ry = sin(rot) * dist;
        const double xi = floor(rx / G.cell_size + half), yi = floor(ry / G.cell_size + half);
        if (!(xi >= 0 && xi < G.cell_num && yi >= 0 && yi < G.cell_num)) continue;     // :134-137 (-inf = outside)
        const int cell = G.cell_num * (int)yi + (int)xi;
        const double vrot = atan2(vj.y, vj.x) - angle;                      // :144-148
        const double speed = sqrt(vj.x * vj.x + vj.y * vj.y);
        sx[cell] += cos(vrot) * speed; sy[cell] += sin(vrot) * speed; cnt[cell] += 1;
    }
    float *o = G.out + idx * (size_t)(cells * C);
    for (int c = 0; c < cells; ++c) {
        const bool occ = cnt[c] > 0;
        const double mx = occ ? sx[c] / cnt[c] : 0.0, my = occ ? sy[c] / cnt[c] : 0.0;
        if (C == 1) o[c] = occ ? 1.f : 0.f;
        else if (C == 2) { o[2 * c] = (float)mx; o[2 * c + 1] = (float)my; }
        else { o[3 * c] = occ ? 1.f : 0.f; o[3 * c + 1] = (float)mx; o[3 * c + 2] = (float)my; }
    }
}

}  // namespace cs

extern "C" int crowdsim_pack_joint(int B, int N, const crowdsim_state *st, int kinematics_unicycle, float *out, void *stream)
{
    if (!st || !out || B < 0 || N < 0) return CROWDSIM_EINVAL;
    if (!st->h_pos || !st->h_vel || !st->h_attr || !st->r_pos || !st->r_vel || !st->r_goal || !st->r_attr) return CROWDSIM_EINVAL;
    if (B == 0 || N == 0) return CROWDSIM_OK;
    cs::PackArgs A; A.B = B; A.N = N; A.unicycle = kinematics_unicycle; A.st = *st; A.out = out;
    const size_t n = (size_t)B * N; const int threads = 128; const int blocks = (int)((n + threads - 1) / threads);
    cs::pack_joint_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(A);
    ++cs::g_launches;
    return (int)cudaGetLastError();
}

extern "C" int crowdsim_lookahead_pack(const crowdsim_params *prm, int B, int N, const crowdsim_state *st,
                                       const double *actions, int A, int kinematics_unicycle,
                                       float *out_states, double *out_reward, void *stream)
{
    if (!prm || !st || !actions || !out_states || !out_reward || B < 0 || N < 1 || A < 1) return CROWDSIM_EINVAL;
    if (N > CROWDSIM_MAX_HUMANS || prm->max_neighbors > CROWDSIM_MAX_NEIGHBORS || !cs::policies_supported(prm)) return CROWDSIM_EUNSUPPORTED;
    if (!st->h_pos || !st->h_vel || !st->h_goal || !st->h_attr || !st->r_pos || !st->r_vel || !st->r_goal || !st->r_attr || !st->g_time) return CROWDSIM_EINVAL;
    if (kinematics_unicycle && !st->r_theta) return CROWDSIM_EINVAL;
    if (B == 0) return CROWDSIM_OK;
    cs::LookArgs G;
    G.k = cs::make_kparams(prm, N);
    G.B = B; G.N = N; G.L = N + 1; G.EPB = cs::envs_per_block(G.L, 128); G.A = A; G.unicycle = kinematics_unicycle;
    G.st = *st; G.actions = actions; G.out_states = out_states; G.out_reward = out_reward;
    const int threads = G.EPB * G.L;
    const int blocks = (B + G.EPB - 1) / G.EPB;
    size_t smem = cs::stage_bytes(G.EPB, G.L, G.k.nb_alloc, threads);
    const bool hlin = prm->human_policy == CROWDSIM_HUMANS_LINEAR;
    smem += (size_t)G.EPB * 48 + (size_t)A * 16 + (size_t)G.EPB * G.L * (hlin ? 16 : 8) + (size_t)A * N * 13 * sizeof(float);
    if (smem > 227 * 1024) return CROWDSIM_EUNSUPPORTED;
    if (smem > 48 * 1024) {
        cudaError_t err = hlin ? cudaFuncSetAttribute(cs::lookahead_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                               : cudaFuncSetAttribute(cs::lookahead_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return (int)err;
    }
    if (hlin) cs::lookahead_kernel<true><<<blocks, threads, smem, (cudaStream_t)stream>>>(G);
    else cs::lookahead_kernel<false><<<blocks, threads, smem, (cudaStream_t)stream>>>(G);
    ++cs::g_launches;
    return (int)cudaGetLastError();
}

extern "C" int crowdsim_lookahead_humans(const crowdsim_params *prm, int B, int N, const crowdsim_state *st,
                                         double *next_h_pos, double *next_h_vel, void *stream)
{
    if (!prm || !st || !next_h_pos || !next_h_vel || B < 0 || N < 1) return CROWDSIM_EINVAL;
    if (N > CROWDSIM_MAX_HUMANS || prm->max_neighbors > CROWDSIM_MAX_NEIGHBORS || !cs::policies_supported(prm)) return CROWDSIM_EUNSUPPORTED;
    if (!st->h_pos || !st->h_vel || !st->h_goal || !st->h_attr || !st->r_pos || !st->r_vel || !st->r_attr) return CROWDSIM_EINVAL;
    if (B == 0) return CROWDSIM_OK;
    cs::NextArgs G;
    G.k = cs::make_kparams(prm, N);
    G.B = B; G.N = N; G.L = N + 1; G.EPB = cs::envs_per_block(G.L, 128); G.st = *st; G.next_pos = next_h_pos; G.next_vel = next_h_vel;
    const int threads = G.EPB * G.L;
    const int blocks = (B + G.EPB - 1) / G.EPB;
    const size_t smem = cs::stage_bytes(G.EPB, G.L, G.k.nb_alloc, threads);
    if (smem > 227 * 1024) return CROWDSIM_EUNSUPPORTED;
    const bool hlin = prm->human_policy == CROWDSIM_HUMANS_LINEAR;
    if (smem > 48 * 1024) {
        cudaError_t err = hlin ? cudaFuncSetAttribute(cs::lookahead_humans_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                               : cudaFuncSetAttribute(cs::lookahead_humans_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return (int)err;
    }
    if (hlin) cs::lookahead_humans_kernel<true><<<blocks, threads, smem, (cudaStream_t)stream>>>(G);
    else cs::lookahead_humans_kernel<false><<<blocks, threads, smem, (cudaStream_t)stream>>>(G);
    ++cs::g_launches;
    return (int)cudaGetLastError();
}

extern "C" int crowdsim_occupancy_maps(int B, int N, const double *h_pos, const double *h_vel, int cell_num, double cell_size,
                                       int channels, float *out, void *stream)
{
    if (!h_pos || !h_vel || !out || B < 0 || N < 2 || cell_num < 1 || !(cell_size > 0) || channels < 1 || channels > 3) return CROWDSIM_EINVAL;
    if (cell_num * cell_num > CS_OM_MAX_CELLS) return CROWDSIM_EUNSUPPORTED;
    if (B == 0) return CROWDSIM_OK;
    cs::OmArgs G; G.B = B; G.N = N; G.cell_num = cell_num; G.channels = channels; G.cell_size = cell_size; G.pos = h_pos; G.vel = h_vel; G.out = out;
    const size_t n = (size_t)B * N; const int threads = 128; const int blocks = (int)((n + threads - 1) / threads);
    cs::occupancy_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(G);
    ++cs::g_launches;
    return (int)cudaGetLastError();
}
