"""numpy front-end of oracle/_build/libcrowdsim_oracle.so (TEST INFRASTRUCTURE, not product code).

Mirrors the C ABI's struct-of-pointers layout on host numpy arrays so tests can run the same call on the
CUDA library and on this CPU restatement and compare array for array. Importable only from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
"""
import ctypes as C
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from crowdnav_b200 import _abi  # noqa: E402  (struct definitions only)

sys.path.insert(0, HERE)
import build as _build  # noqa: E402

_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(HERE, '_build', 'libcrowdsim_oracle.so')
        if not os.path.exists(so):
            _build.build()
        l = C.CDLL(so)
        _abi.declare(l, prefix='oracle_crowdsim_', with_stream=False)
        l.oracle_mt19937_doubles.argtypes = [C.c_uint32, C.c_int, C.c_void_p]
        l.oracle_get_stats.argtypes = [C.c_void_p]
        l.oracle_crowdsim_run_passes.restype = C.c_int
        l.oracle_crowdsim_run_passes.argtypes = [C.POINTER(_abi.Params), C.c_int, C.c_int, C.POINTER(_abi.State),
                                                 C.POINTER(_abi.StepIO), C.POINTER(_abi.ResetArgs), C.c_int]
        _lib = l
    return _lib


def default_params(**over):
    p = dict(time_step=0.25, time_limit=25.0, success_reward=1.0, collision_penalty=-0.25, discomfort_dist=0.2,
             discomfort_penalty_factor=0.5, neighbor_dist=10.0, time_horizon=5.0, max_neighbors=10,
             human_safety_space=0.0, robot_safety_space=0.0, robot_visible=0, robot_policy=_abi.ROBOT_ORCA)
    p.update(over)
    return _abi.Params(**p)


def _ptr(a):
    return None if a is None else a.ctypes.data


class HostState(object):
    """B envs x N humans on host numpy arrays, same layout as crowdsim_state."""

    def __init__(self, B, N, with_active=True):
        self.B, self.N = B, N
        z = lambda *s: np.zeros(s, dtype=np.float64)  # noqa: E731
        self.h_pos, self.h_vel, self.h_goal, self.h_attr = z(B, N, 2), z(B, N, 2), z(B, N, 2), z(B, N, 2)
        self.r_pos, self.r_vel, self.r_goal, self.r_attr = z(B, 2), z(B, 2), z(B, 2), z(B, 2)
        self.r_theta, self.g_time = z(B), z(B)
        self.active = np.ones(B, dtype=np.uint8) if with_active else None

    FIELDS = ('h_pos', 'h_vel', 'h_goal', 'h_attr', 'r_pos', 'r_vel', 'r_goal', 'r_attr', 'r_theta', 'g_time')

    def struct(self):
        return _abi.State(*[_ptr(getattr(self, f)) for f in self.FIELDS], _ptr(self.active))

    def copy(self):
        o = HostState(self.B, self.N, self.active is not None)
        for f in self.FIELDS:
            getattr(o, f)[...] = getattr(self, f)
        if self.active is not None:
            o.active[...] = self.active
        return o

    def set_scene(self, e, scene):
        """scene = {'robot': [px,py,vx,vy,gx,gy,r,vpref,theta], 'humans': [[px,py,vx,vy,gx,gy,r,vpref],..]}"""
        r = [float(x) for x in scene['robot']]
        self.r_pos[e] = r[0:2]; self.r_vel[e] = r[2:4]; self.r_goal[e] = r[4:6]; self.r_attr[e] = r[6:8]
        self.r_theta[e] = r[8]
        for i, h in enumerate(scene['humans']):
            h = [float(x) for x in h]
            self.h_pos[e, i] = h[0:2]; self.h_vel[e, i] = h[2:4]; self.h_goal[e, i] = h[4:6]; self.h_attr[e, i] = h[6:8]
        for i in range(len(scene['humans']), self.N):      # `mixed` scenes with fewer humans: park the unused slots
            x = _abi.PARKED_X + 100.0 * i
            self.h_pos[e, i] = (x, _abi.PARKED_X); self.h_vel[e, i] = 0.0; self.h_goal[e, i] = (x, _abi.PARKED_X)
            self.h_attr[e, i] = (0.3, 1.0)


class HostStepIO(object):
    def __init__(self, B):
        self.action = np.zeros((B, 2)); self.action_out = np.zeros((B, 2))
        self.reward = np.zeros(B); self.dmin = np.zeros(B)
        self.done = np.zeros(B, dtype=np.uint8); self.info = np.zeros(B, dtype=np.uint8)

    def struct(self):
        return _abi.StepIO(_ptr(self.action), _ptr(self.action_out), _ptr(self.reward), _ptr(self.dmin),
                           _ptr(self.done), _ptr(self.info))


def discount_table(gamma, time_step, v_pref, n=128):
    """explorer.py:71-72: pow(gamma, t * time_step * v_pref), with C/Python pow."""
    return np.array([pow(gamma, t * time_step * v_pref) for t in range(n)], dtype=np.float64)


class HostEpisodes(object):
    def __init__(self, B, k, gamma=0.9, time_step=0.25, v_pref=1.0, max_steps=128):
        """max_steps: length of the discount table, at least the longest episode (steps beyond it count as undiscounted
        to zero, like the kernels do)."""
        self.ep_case = np.full(B, -1, dtype=np.int32); self.ep_steps = np.zeros(B, dtype=np.int32)
        self.ep_return = np.zeros(B); self.ep_too_close = np.zeros(B, dtype=np.int32)
        self.ep_min_dist_sum = np.zeros(B)
        self.discount = discount_table(gamma, time_step, v_pref, max(128, max_steps))
        self.res_info = np.zeros(k, dtype=np.uint8); self.res_steps = np.zeros(k, dtype=np.int32)
        self.res_time = np.zeros(k); self.res_return = np.zeros(k)
        self.res_too_close = np.zeros(k, dtype=np.int32); self.res_min_dist_sum = np.zeros(k)
        self.res_final_rpos = np.zeros((k, 2))

    def struct(self):
        return _abi.Episodes(_ptr(self.ep_case), _ptr(self.ep_steps), _ptr(self.ep_return), _ptr(self.ep_too_close),
                             _ptr(self.ep_min_dist_sum), _ptr(self.discount), len(self.discount),
                             _ptr(self.res_info), _ptr(self.res_steps), _ptr(self.res_time), _ptr(self.res_return),
                             _ptr(self.res_too_close), _ptr(self.res_min_dist_sum), _ptr(self.res_final_rpos))


class HostAutoReset(object):
    """crowdsim_autoreset on host arrays (next-scene slot per env)."""

    def __init__(self, B, N, circle_radius=4.0, robot_radius=0.3, robot_v_pref=1.0):
        self.n_h_pos = np.zeros((B, N, 2)); self.n_h_goal = np.zeros((B, N, 2)); self.n_h_attr = np.zeros((B, N, 2))
        self.n_case = np.full(B, -1, dtype=np.int32)
        self.n_state = np.zeros(B, dtype=np.uint8); self.want = np.zeros(B, dtype=np.uint8)
        self.circle_radius, self.robot_radius, self.robot_v_pref = circle_radius, robot_radius, robot_v_pref

    def struct(self):
        return _abi.AutoReset(_ptr(self.n_h_pos), _ptr(self.n_h_goal), _ptr(self.n_h_attr), _ptr(self.n_case),
                              _ptr(self.n_state), _ptr(self.want), self.circle_radius, self.robot_radius, self.robot_v_pref)


def _reset_args(seeds, rule, mask, circle_radius, square_width, human_radius, human_v_pref, robot_radius, robot_v_pref,
                discomfort_dist, randomize_attributes, seed_stride, case_counter, case_total, seed_base, case_first=0, case_wrap=0):
    return _abi.ResetArgs(_ptr(mask), _ptr(seeds), int(seed_stride), _abi.RULES[rule], circle_radius, square_width,
                          human_radius, human_v_pref, robot_radius, robot_v_pref, discomfort_dist,
                          int(randomize_attributes), _ptr(case_counter), int(case_total), int(seed_base), int(case_first), int(case_wrap))


def prefetch(ar, B, N, seeds=None, rule='circle_crossing', circle_radius=4.0, square_width=10.0, human_radius=0.3,
             human_v_pref=1.0, robot_radius=0.3, robot_v_pref=1.0, discomfort_dist=0.2, randomize_attributes=False,
             seed_stride=0, case_counter=None, case_total=0, seed_base=0):
    a = _reset_args(seeds, rule, None, circle_radius, square_width, human_radius, human_v_pref, robot_radius,
                    robot_v_pref, discomfort_dist, randomize_attributes, seed_stride, case_counter, case_total, seed_base)
    s = ar.struct()
    rc = lib().oracle_crowdsim_prefetch_scenes(C.byref(a), B, N, C.byref(s))
    assert rc == 0, rc


def reset(st, seeds, rule='circle_crossing', mask=None, ep=None, circle_radius=4.0, square_width=10.0,
          human_radius=0.3, human_v_pref=1.0, robot_radius=0.3, robot_v_pref=1.0, discomfort_dist=0.2,
          randomize_attributes=False, seed_stride=0, case_counter=None, case_total=0, seed_base=0):
    """seeds: uint32 array; with seed_stride != 0 it must be a writable contiguous uint32 array (advanced in place)."""
    if seeds is not None and not (isinstance(seeds, np.ndarray) and seeds.dtype == np.uint32 and seeds.flags['C_CONTIGUOUS']):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
    mask = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
    a = _reset_args(seeds, rule, mask, circle_radius, square_width, human_radius, human_v_pref, robot_radius,
                    robot_v_pref, discomfort_dist, randomize_attributes, seed_stride, case_counter, case_total, seed_base)
    s = st.struct(); e = ep.struct() if ep is not None else None
    rc = lib().oracle_crowdsim_reset(C.byref(a), st.B, st.N, C.byref(s), C.byref(e) if e is not None else None)
    assert rc == 0, rc


def step(prm, st, io, ep=None, ar=None):
    s, i = st.struct(), io.struct(); e = ep.struct() if ep is not None else None
    a = ar.struct() if ar is not None else None
    rc = lib().oracle_crowdsim_step(C.byref(prm), st.B, st.N, C.byref(s), C.byref(i),
                                    C.byref(e) if e is not None else None, C.byref(a) if a is not None else None)
    assert rc == 0, rc


def run_passes(prm, st, io, seeds, n_passes, rule='circle_crossing', seed_stride=0, circle_radius=4.0, square_width=10.0,
               human_radius=0.3, human_v_pref=1.0, robot_radius=0.3, robot_v_pref=1.0, discomfort_dist=0.2,
               randomize_attributes=False):
    """n_passes x (step; reset of the envs whose episode ended, from the per-slot seeds) inside one C call / one OpenMP
    parallel region. `seeds` (uint32 [B]) is advanced in place by seed_stride per use, like reset(..., seed_stride=...)."""
    assert isinstance(seeds, np.ndarray) and seeds.dtype == np.uint32 and seeds.flags['C_CONTIGUOUS']
    a = _reset_args(seeds, rule, None, circle_radius, square_width, human_radius, human_v_pref, robot_radius,
                    robot_v_pref, discomfort_dist, randomize_attributes, seed_stride, None, 0, 0)
    s, i = st.struct(), io.struct()
    rc = lib().oracle_crowdsim_run_passes(C.byref(prm), st.B, st.N, C.byref(s), C.byref(i), C.byref(a), int(n_passes))
    _abi.check(rc, 'oracle_crowdsim_run_passes')


def orca_act(prm, st):
    out = np.zeros((st.B, 2)); s = st.struct()
    rc = lib().oracle_crowdsim_orca_act(C.byref(prm), st.B, st.N, C.byref(s), _ptr(out))
    assert rc == 0, rc
    return out


def pack_joint(st, unicycle=False):
    out = np.zeros((st.B, st.N, 13), dtype=np.float32); s = st.struct()
    rc = lib().oracle_crowdsim_pack_joint(st.B, st.N, C.byref(s), int(unicycle), _ptr(out))
    assert rc == 0, rc
    return out


def lookahead_pack(prm, st, actions, unicycle=False):
    actions = np.ascontiguousarray(actions, dtype=np.float64); A = actions.shape[0]
    states = np.zeros((st.B, A, st.N, 13), dtype=np.float32); reward = np.zeros((st.B, A)); s = st.struct()
    rc = lib().oracle_crowdsim_lookahead_pack(C.byref(prm), st.B, st.N, C.byref(s), _ptr(actions), A, int(unicycle),
                                              _ptr(states), _ptr(reward))
    assert rc == 0, rc
    return states, reward


def mt19937_doubles(seed, n):
    out = np.zeros(n); lib().oracle_mt19937_doubles(seed, n, _ptr(out)); return out


def set_threads(n):
    lib().oracle_set_threads(int(n))


def max_threads():
    return int(lib().oracle_get_max_threads())


def get_stats():
    out = (C.c_long * 4)(); lib().oracle_get_stats(out); return tuple(out)


def run_episodes(prm, N, seeds, rule='circle_crossing', gamma=0.9, robot_v_pref=1.0, max_steps=200, **reset_kw):
    """Run one episode per seed to termination (lockstep, finished envs frozen); returns HostEpisodes + state."""
    B = len(seeds)
    st = HostState(B, N); io = HostStepIO(B); ep = HostEpisodes(B, B, gamma, prm.time_step, robot_v_pref, max_steps)
    ep.ep_case[:] = np.arange(B)
    reset(st, seeds, rule, ep=ep, robot_v_pref=robot_v_pref, **reset_kw)
    for _ in range(max_steps):
        if not st.active.any():
            break
        step(prm, st, io, ep)
    assert not st.active.any()
    return ep, st


def occupancy_maps(h_pos, h_vel, cell_num=4, cell_size=1.0, channels=3):
    """MultiHumanRL.build_occupancy_maps (crowd_nav/policy/multi_human_rl.py:109-163) restated for [B][N][2] float64
    position / velocity arrays -> [B][N][cell_num^2 * channels] float32. Plain float64 loops in the reference's
    expression order (rotation into the human's velocity frame :121-129, floor to cell indices :132-138, per-cell mean
    of the occupants' rotated velocities :143-160)."""
    import math
    h_pos = np.asarray(h_pos, dtype=np.float64); h_vel = np.asarray(h_vel, dtype=np.float64)
    B, N = h_pos.shape[:2]
    if N < 2:
        raise ValueError('need at least one array to concatenate')
    cells = cell_num * cell_num
    out = np.zeros((B, N, cells * channels), dtype=np.float32)
    for e in range(B):
        for i in range(N):
            angle = math.atan2(h_vel[e, i, 1], h_vel[e, i, 0])
            lists = [([], []) for _ in range(cells)]
            for j in range(N):
                if j == i:
                    continue
                ox = h_pos[e, j, 0] - h_pos[e, i, 0]; oy = h_pos[e, j, 1] - h_pos[e, i, 1]
                rot = math.atan2(oy, ox) - angle
                dist = math.sqrt(ox * ox + oy * oy)
                rx = math.cos(rot) * dist; ry = math.sin(rot) * dist
                xi = math.floor(rx / cell_size + cell_num / 2); yi = math.floor(ry / cell_size + cell_num / 2)
                if xi < 0 or xi >= cell_num or yi < 0 or yi >= cell_num:
                    continue
                vrot = math.atan2(h_vel[e, j, 1], h_vel[e, j, 0]) - angle
                speed = math.sqrt(h_vel[e, j, 0] * h_vel[e, j, 0] + h_vel[e, j, 1] * h_vel[e, j, 1])
                lists[cell_num * yi + xi][0].append(math.cos(vrot) * speed)
                lists[cell_num * yi + xi][1].append(math.sin(vrot) * speed)
            for c, (lx, ly) in enumerate(lists):
                occ = len(lx) > 0
                mx = sum(lx) / len(lx) if occ else 0.0
                my = sum(ly) / len(ly) if occ else 0.0
                if channels == 1:
                    out[e, i, c] = 1.0 if occ else 0.0
                elif channels == 2:
                    out[e, i, 2 * c] = mx; out[e, i, 2 * c + 1] = my
                else:
                    out[e, i, 3 * c] = 1.0 if occ else 0.0; out[e, i, 3 * c + 1] = mx; out[e, i, 3 * c + 2] = my
    return out


def lookahead_humans(prm, st):
    """The observation of env.onestep_lookahead (crowd_sim.py:414-416): one oracle step on a COPY of the state; the
    humans' next states do not depend on the robot's action."""
    cp = st.copy()
    io = HostStepIO(st.B)
    step(prm, cp, io)
    return cp.h_pos.copy(), cp.h_vel.copy()
