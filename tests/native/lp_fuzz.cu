// lp_fuzz.cu -- CPU fuzz test (test infrastructure): the CUDA solver's arithmetic compiled FOR THE HOST
// (crowdnav_b200/csrc/orca_device.cuh, orca_spec.cuh are __host__ __device__) against the C oracle
// (oracle/rvo2_f32.h) on millions of random ORCA problems, bit for bit:
//   A  make_line / make_line_sel / make_line_far + make_line_overlap   vs  orc_make_line, time horizon and time step drawn
//      per case from {5, 3, 2.5, 10} s and {0.25, 0.1, 0.2, 1/30} s
//   B  sequential lp2 + lp3 (shared-memory-column code path of the generic kernel, n <= 10)   vs  orc_lp2 / orc_lp3
//   C  speculative lp1_all + lp2_scan (register path of the small-crowd kernel, n <= 5)        vs  orc_lp2
//   D  lp3 as independent per-line sub-problems + lp3_outer_scan (the lane-parallel pass)      vs  orc_lp3
//   F  lp3 on lanes: (i, j) pair projections + speculative per-line sub-problems (lp3_project_pair, lp3_sub_spec<4> and <9>)
//      + lp3_outer_scan                                                                        vs  orc_lp3
//   H  insert_sorted<10> (sorted register list of the crowd kernel, 20-60 candidates incl. ties) vs  orc_insert_neighbor
//   E  neighbour_order (pair-wise ranks + packed indices of the small-crowd kernel)            vs  orc_insert_neighbor
// Build (tests/test_native_cpu.py): nvcc -O2 --fmad=false -Xcompiler -ffp-contract=off -std=c++17 lp_fuzz.cu
// Usage: lp_fuzz <cases> <seed>; prints coverage counters; exit code 0 iff every comparison was bit-identical.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdint>
#include <type_traits>
#include "../../crowdnav_b200/csrc/orca_device.cuh"
#include "../../crowdnav_b200/csrc/orca_spec.cuh"
extern "C" {
#include "../../oracle/rvo2_f32.h"
}

static uint64_t rng_state;
static inline uint32_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (uint32_t)(rng_state >> 16); }
static inline float uni(float a, float b) { return a + (b - a) * (rnd() / 4294967296.0f); }
static inline bool same(float a, float b) { return memcmp(&a, &b, 4) == 0; }

template <int M>
static bool check_case(int n, const orc_line *ol, float radius, orc_v2 opt, long *cov)
{
    using namespace orca;
    // ---- oracle ----
    orc_v2 ores; const int ofail = orc_lp2(ol, n, radius, opt, 0, &ores);
    orc_v2 ores3 = ores; if (ofail < n) orc_lp3(ol, n, ofail, radius, &ores3);
    cov[0] += (ofail < n);
    // ---- B: sequential code on column-layout arrays (stride 1) ----
    float lbuf[4 * 16], pbuf[4 * 16];
    const Lines L = { lbuf, 1 }, P = { pbuf, 1 };
    for (int k = 0; k < n; ++k) L.set(k, mk(ol[k].point.x, ol[k].point.y), mk(ol[k].dir.x, ol[k].dir.y));
    V2 r; const int f = lp2(L, n, radius, mk(opt.x, opt.y), false, r);
    if (f != ofail || !same(r.x, ores.x) || !same(r.y, ores.y)) { printf("B lp2 mismatch n=%d\n", n); return false; }
    V2 r3 = r; if (f < n) lp3(L, n, f, radius, P, r3);
    if (!same(r3.x, ores3.x) || !same(r3.y, ores3.y)) { printf("B lp3 mismatch n=%d fail=%d\n", n, f); return false; }
    // ---- D: lp3 as independent sub-problems + outer scan ----
    if (f < n) {
        V2 sub_r[16]; bool sub_ok[16];
        for (int i = 1; i < n; ++i) sub_ok[i] = lp3_subproblem(L, i, radius, P, sub_r[i]);
        V2 rd = r;
        lp3_outer_scan(L, n, f, radius, rd, [&](int ii, V2 &r2) { r2 = sub_r[ii]; return sub_ok[ii]; });
        if (!same(rd.x, ores3.x) || !same(rd.y, ores3.y)) { printf("D lp3 sub-problem mismatch n=%d fail=%d\n", n, f); return false; }
    }
    // ---- F: the lane-parallel pass of the kernels: every (i, j) projection on its own, every sub-problem speculative ----
    if (f < n) {
        V2 sub_r[16]; bool sub_ok[16];
        auto run = [&](auto kc) {
            constexpr int K = decltype(kc)::value;
            for (int i = 1; i < n; ++i) {
                RegLines<K> Pr; bool pv[K];
                for (int j = 0; j < K; ++j) {
                    Pr.p[j] = mk(0.f, 0.f); Pr.d[j] = mk(0.f, 0.f); pv[j] = false;
                    if (j < i) pv[j] = lp3_project_pair(L.point(i), L.dir(i), L.point(j), L.dir(j), Pr.p[j], Pr.d[j]);
                }
                sub_ok[i] = lp3_sub_spec<K>(Pr, pv, radius, L.dir(i), sub_r[i]);
            }
            V2 rd = r;
            lp3_outer_scan(L, n, f, radius, rd, [&](int ii, V2 &r2) { r2 = sub_r[ii]; return sub_ok[ii]; });
            return same(rd.x, ores3.x) && same(rd.y, ores3.y);
        };
        if (n <= 5 && !run(std::integral_constant<int, 4>())) { printf("F lane-parallel lp3 (K=4) mismatch n=%d fail=%d\n", n, f); return false; }
        if (!run(std::integral_constant<int, 9>())) { printf("F lane-parallel lp3 (K=9) mismatch n=%d fail=%d\n", n, f); return false; }
        cov[6]++;
    }
    // ---- C: speculative register path (n <= M) ----
    if (n <= M) {
        RegLines<M> R; bool valid[M];
        for (int k = 0; k < M; ++k) { valid[k] = k < n; R.p[k] = k < n ? mk(ol[k].point.x, ol[k].point.y) : mk(0, 0); R.d[k] = k < n ? mk(ol[k].dir.x, ol[k].dir.y) : mk(0, 0); }
        V2 cand[M]; bool feas[M];
        lp1_all<M, M>(R, valid, radius, mk(opt.x, opt.y), false, cand, feas);
        V2 rs; const int fs = lp2_scan<M, M>(R, valid, n, cand, feas, lp2_init(mk(opt.x, opt.y), radius), rs);
        if (fs != ofail || !same(rs.x, ores.x) || !same(rs.y, ores.y)) { printf("C speculative lp2 mismatch n=%d (fail %d vs %d)\n", n, fs, ofail); return false; }
        cov[1]++;
    }
    return true;
}

// ---- E: M candidates in scan order, some out of range, many exact ties: order and count must equal RVO2's insertion sort
// (neighbour range 10 m, capacity max_nb >= M as in the small-crowd kernel's callers; truncation to max_nb < M keeps the
// first max_nb entries of the same order) ----
template <int M>
static bool check_order(long *cov)
{
    float dsq[M]; bool inr[M]; int id[M], src[M];
    const float range_sq = 100.0f;
    const bool ties = rnd() % 3 == 0;
    for (int c = 0; c < M; ++c) {
        const float x = ties ? (float)(rnd() % 4) * 0.5f : uni(-9.f, 9.f), y = ties ? (float)(rnd() % 3) : uni(-9.f, 9.f);
        dsq[c] = x * x + y * y;
        const bool visible = (rnd() % 8) != 0;                 // e.g. the invisible robot's slot
        inr[c] = visible && dsq[c] < range_sq;
        id[c] = (c + (int)(rnd() % 2)) % 6;                    // agent indices < 8, not necessarily ascending
    }
    const int nl = orca::neighbour_order<M>(dsq, inr, id, src);
    float nd[M]; int ni[M]; int cnt = 0; float rs = range_sq;
    for (int c = 0; c < M; ++c) if (inr[c]) orc_insert_neighbor(dsq[c], id[c], nd, ni, &cnt, M, &rs);
    if (nl != cnt) { printf("E count mismatch %d vs %d\n", nl, cnt); return false; }
    for (int kk = 0; kk < M; ++kk) {
        const int want = kk < cnt ? ni[kk] : 0;
        if (src[kk] != want) { printf("E order mismatch at %d: %d vs %d (M=%d)\n", kk, src[kk], want, M); return false; }
    }
    cov[4] += 1; cov[5] += ties;
    return true;
}

// ---- H: the crowd kernel's neighbour list: n candidates (some out of range, many exact ties), capacity 10 and smaller ----
static bool check_sorted_insert(long *cov)
{
    constexpr int M = 10;
    const int n = 1 + rnd() % 63, max_nb = (rnd() % 4 == 0) ? 1 + (int)(rnd() % 10) : 10;
    const float range_sq = 100.0f, inf = __builtin_inff();
    const bool ties = rnd() % 3 == 0;
    float td[M]; int tj[M]; for (int k = 0; k < M; ++k) { td[k] = inf; tj[k] = 0; }
    float nd[M]; int ni[M]; int cnt = 0; float rs = range_sq; int in_range = 0;
    for (int j = 0; j < n; ++j) {
        const float x = ties ? (float)(rnd() % 5) * 0.5f : uni(-11.f, 11.f), y = ties ? (float)(rnd() % 4) : uni(-11.f, 11.f);
        const float d = x * x + y * y;
        const bool in = (rnd() % 10 != 0) && d < range_sq;
        orca::insert_sorted<M>(in ? d : inf, j, td, tj);
        in_range += in;
        if (in) orc_insert_neighbor(d, j, nd, ni, &cnt, max_nb, &rs);
    }
    int nl = in_range < max_nb ? in_range : max_nb;
    if (nl != cnt) { printf("H count mismatch %d vs %d\n", nl, cnt); return false; }
    for (int k = 0; k < nl; ++k) if (tj[k] != ni[k] || !same(td[k], nd[k])) { printf("H order mismatch at %d (n=%d max_nb=%d)\n", k, n, max_nb); return false; }
    cov[7] += 1;
    return true;
}

int main(int argc, char **argv)
{
    const long cases = argc > 1 ? atol(argv[1]) : 200000;
    rng_state = argc > 2 ? strtoull(argv[2], nullptr, 10) * 2654435761ull + 88172645463325252ull : 88172645463325252ull;
    long cov[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    using namespace orca;
    for (int i = 1, q = 0; i <= 9; ++i) for (int j = 0; j < i; ++j, ++q) { int a, b; lp3_pair_of(q, a, b); if (a != i || b != j) { printf("lp3_pair_of(%d)\n", q); return 1; } }
    for (long c = 0; c < cases; ++c) {
        const int kind = rnd() % 4;
        const int n = 1 + rnd() % ((kind == 3) ? 10 : 5);
        orc_line ol[16];
        const float radius = uni(0.5f, 1.5f);
        orc_v2 opt = orc_mk(uni(-1.2f, 1.2f), uni(-1.2f, 1.2f));
        // time horizon and time step of the env's config (default 5 s / 0.25 s; 0.1, 0.2 and 1/30 are not powers of two),
        // converted the way the kernels' launch set-up does (crowdsim_common.cuh): inverses of the float32 values
        static const double horizons[4] = {5.0, 3.0, 2.5, 10.0}, steps[4] = {0.25, 0.1, 0.2, 1.0 / 30.0};
        const int hsel = rnd() % 4, tsel = rnd() % 4;
        const float th = (float)horizons[hsel], dt = (float)steps[tsel];
        const float inv_th = 1.0f / th, inv_dt = 1.0f / dt;
        cov[8] += (hsel != 0); cov[9] += (tsel != 0);
        if (kind <= 1 || kind == 3) {
            // lines from a random crowd around an agent at the origin (kind 1: tight -> overlaps, infeasible LPs)
            const float spread = (kind == 1) ? 1.0f : 4.0f;
            const orc_v2 p = orc_mk(0.f, 0.f), v = orc_mk(uni(-1, 1), uni(-1, 1));
            for (int k = 0; k < n; ++k) {
                const orc_v2 po = orc_mk(uni(-spread, spread), uni(-spread, spread)), vo = orc_mk(uni(-1, 1), uni(-1, 1));
                const float r = uni(0.2f, 0.5f), ro = uni(0.2f, 0.5f);
                ol[k] = orc_make_line(p, v, r, po, vo, ro, inv_th, dt);
                // ---- A: line construction ----
                V2 lp, ld, sp, sd;
                make_line(mk(p.x, p.y), mk(v.x, v.y), r, mk(po.x, po.y), mk(vo.x, vo.y), ro, inv_th, inv_dt, lp, ld);
                make_line_sel(mk(p.x, p.y), mk(v.x, v.y), r, mk(po.x, po.y), mk(vo.x, vo.y), ro, inv_th, inv_dt, sp, sd);
                {   // straight-line form + overlap repair (multi-step kernel)
                    V2 fp, fd; bool ov;
                    make_line_far(mk(p.x, p.y), mk(v.x, v.y), r, mk(po.x, po.y), mk(vo.x, vo.y), ro, inv_th, fp, fd, ov);
                    if (ov) make_line_overlap(mk(p.x, p.y), mk(v.x, v.y), r, mk(po.x, po.y), mk(vo.x, vo.y), ro, inv_dt, fp, fd);
                    if (!same(fp.x, lp.x) || !same(fp.y, lp.y) || !same(fd.x, ld.x) || !same(fd.y, ld.y)) { printf("A far/overlap line mismatch\n"); return 1; }
                }
                if (!same(lp.x, ol[k].point.x) || !same(lp.y, ol[k].point.y) || !same(ld.x, ol[k].dir.x) || !same(ld.y, ol[k].dir.y) ||
                    !same(sp.x, lp.x) || !same(sp.y, lp.y) || !same(sd.x, ld.x) || !same(sd.y, ld.y)) { printf("A line mismatch\n"); return 1; }
                const float dsq = po.x * po.x + po.y * po.y; cov[2] += (dsq <= (r + ro) * (r + ro));
            }
        } else {
            // adversarial: arbitrary half-planes incl. exactly parallel / anti-parallel / duplicated lines and far-away points
            for (int k = 0; k < n; ++k) {
                const float ang = uni(-3.2f, 3.2f);
                ol[k].dir = orc_mk(cosf(ang), sinf(ang));
                ol[k].point = orc_mk(uni(-2, 2), uni(-2, 2));
                if (k > 0 && rnd() % 4 == 0) { ol[k].dir = ol[rnd() % k].dir; cov[3]++; }
                if (k > 0 && rnd() % 6 == 0) { const orc_v2 d = ol[rnd() % k].dir; ol[k].dir = orc_mk(-d.x, -d.y); cov[3]++; }
                if (k > 0 && rnd() % 12 == 0) ol[k] = ol[rnd() % k];
            }
        }
        if (!check_case<5>(n, ol, radius, opt, cov)) { printf("case %ld kind %d\n", c, kind); return 1; }
        if (n > 5) { long dummy[8] = {0}; if (!check_case<10>(n, ol, radius, opt, dummy)) { printf("case %ld kind %d (M = 10)\n", c, kind); return 1; } cov[1] += dummy[1]; }
        if (!check_sorted_insert(cov)) { printf("case %ld\n", c); return 1; }
        if (!(check_order<5>(cov) && check_order<4>(cov) && check_order<2>(cov) && check_order<1>(cov))) { printf("case %ld\n", c); return 1; }
    }
    printf("ok cases=%ld lp3_needed=%ld speculative_checked=%ld overlapping_pairs=%ld forced_parallel_lines=%ld neighbour_orders=%ld neighbour_ties=%ld lane_lp3_checked=%ld sorted_lists=%ld other_horizon=%ld other_time_step=%ld\n", cases, cov[0], cov[1], cov[2], cov[3], cov[4], cov[5], cov[6], cov[7], cov[8], cov[9]);
    return 0;
}
