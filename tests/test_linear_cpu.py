"""CPU tests of the Linear policy (env.config [humans] policy = linear, test.py --policy linear): argument validation of the
library without a GPU, the C oracle with the Linear policy (tests/native/linear_oracle.c) against the reference's own
fixtures (tests/golden/*linear*), the `mixed` quirks, and the regeneration of those fixtures from the reference."""
import ctypes as C
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import linear_oracle as lin
from linear_suites import LINEAR_SUITES, TOL, params
from util import load_golden, scene_arrays, fill_host_state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = '/root/reference'


def test_unknown_policy_is_rejected_before_any_launch():
    from crowdnav_b200 import build, _abi
    build.build()
    lib = _abi.load()
    n0 = lib.crowdsim_launch_count()
    dummy = C.c_void_p(16)                 # never dereferenced: the policy check comes first
    st, io = _abi.State(), _abi.StepIO()
    for over in (dict(human_policy=2), dict(human_policy=-1), dict(robot_policy=4), dict(robot_policy=-1)):
        prm = _abi.Params(0.25, 25.0, 1.0, -0.25, 0.2, 0.5, 10.0, 5.0, 10, 0.0, 0.0, 0, _abi.ROBOT_ORCA)
        for k, v in over.items():
            setattr(prm, k, v)
        assert lib.crowdsim_step(C.byref(prm), 1, 5, C.byref(st), C.byref(io), None, None, None) == -2, over
        assert lib.crowdsim_step_n(C.byref(prm), 1, 5, C.byref(st), C.byref(io), None, None, 4, None) == -2, over
        assert lib.crowdsim_onestep_lookahead(C.byref(prm), 1, 5, C.byref(st), C.byref(io), dummy, dummy, None) == -2, over
        assert lib.crowdsim_orca_act(C.byref(prm), 1, 5, C.byref(st), dummy, None) == -2, over
        assert lib.crowdsim_lookahead_pack(C.byref(prm), 1, 5, C.byref(st), dummy, 81, 0, dummy, dummy, None) == -2, over
        assert lib.crowdsim_lookahead_humans(C.byref(prm), 1, 5, C.byref(st), dummy, dummy, None) == -2, over
        assert lib.crowdsim_human_times(C.byref(prm), 1, 5, C.byref(st), dummy, dummy, None, 10, None) == -2, over
    assert lib.crowdsim_launch_count() == n0
    # the 13-argument positional form still means ORCA humans
    assert _abi.Params(0.25, 25.0, 1.0, -0.25, 0.2, 0.5, 10.0, 5.0, 10, 0.0, 0.0, 0, _abi.ROBOT_LINEAR).human_policy == _abi.HUMANS_ORCA


def test_oracle_rejects_unknown_policy(oracle):
    st, io = oracle.HostState(1, 5), oracle.HostStepIO(1)
    for prm in (oracle.default_params(human_policy=5), oracle.default_params(robot_policy=7)):
        assert lin.step_rc(prm, st, io) == -2


def test_configure_accepts_linear_humans_only():
    """BatchedCrowdSim.configure without a device: the config check runs before any allocation."""
    from crowdnav_b200 import _abi
    from crowdnav_b200.batched import BatchedCrowdSim, default_config
    env = BatchedCrowdSim.__new__(BatchedCrowdSim)
    env.B, env.device = 1, 'cpu'
    env._alloc = lambda: None
    for pol in ('orca', 'linear'):
        BatchedCrowdSim.configure(env, default_config(human_policy=pol))
        assert env.human_policy == _abi.HUMAN_POLICIES[pol]
    env.robot_policy, env.robot_visible = _abi.ROBOT_ORCA, False
    env.neighbor_dist, env.time_horizon, env.max_neighbors = 10.0, 5.0, 10
    env.human_safety_space = env.robot_safety_space = 0.0
    assert env.params().human_policy == _abi.HUMANS_LINEAR
    BatchedCrowdSim.set_robot_policy(env, 'linear')
    assert env.params().robot_policy == _abi.ROBOT_LINEAR and env.robot_decides_on_device()
    with pytest.raises(NotImplementedError):
        BatchedCrowdSim.configure(env, default_config(human_policy='sarl'))


@pytest.mark.parametrize('name', sorted(LINEAR_SUITES))
def test_oracle_reproduces_linear_suites(oracle, name):
    """Every case of the reference's suite: terminal class and step count identical; time, discounted return, danger
    statistics and the final positions within TOL. Final velocities: see test_final_velocity_bar."""
    N, rule, _, _, _ = LINEAR_SUITES[name]
    cases = load_golden('suite_' + name)['cases']
    ep, st = lin.run_episodes(params(oracle, name), N, [1000 + c['case'] for c in cases], rule)
    for i, c in enumerate(cases):
        assert ep.res_info[i] == c['info'] and ep.res_steps[i] == c['steps'], c['case']
        assert abs(ep.res_time[i] - (25.0 if c['info'] == 4 else float(c['global_time']))) <= TOL
        assert abs(ep.res_return[i] - float(c['return'])) <= TOL
        assert ep.res_too_close[i] == c['too_close']
        assert abs(ep.res_min_dist_sum[i] - float(c['min_dist_sum'])) <= TOL
        r, h = scene_arrays(c['final'], N)
        assert np.abs(ep.res_final_rpos[i] - r[:2]).max() <= TOL, c['case']
        assert np.abs(st.h_pos[i] - h[:, :2]).max() <= TOL, c['case']
        assert np.abs(st.h_vel[i] - h[:, 2:4]).max() <= 1e-11, c['case']


def test_final_velocity_bar(oracle):
    """The one place a whole-episode comparison needs more than TOL: a linear human that has passed its goal oscillates
    around it, and its direction is that of a vector shorter than a step, so a position difference of a few 1e-13 (the
    1-ulp arctan2 differences, summed over the episode) becomes a larger velocity difference. Measured: square20 case 94,
    4.7e-13 in a position -> 1.9e-12 in a velocity; every recorded single step stays within TOL (test below)."""
    name, N = 'square20_linear_humans', 20
    c = load_golden('suite_' + name)['cases'][94]
    ep, st = lin.run_episodes(params(oracle, name), N, [1000 + 94], 'square_crossing')
    r, h = scene_arrays(c['final'], N)
    dp, dv = np.abs(st.h_pos[0] - h[:, :2]).max(axis=1), np.abs(st.h_vel[0] - h[:, 2:4]).max(axis=1)
    j = int(np.argmax(dv))
    assert dv[j] > TOL and dp[j] <= TOL
    assert np.hypot(*(h[j, :2] - h[j, 4:6])) < 0.25 + 1e-9          # the human is within one step of its goal


@pytest.mark.parametrize('name', sorted(LINEAR_SUITES))
def test_oracle_steps_reproduce_linear_trajectories(oracle, name):
    """Every recorded step of the reference's trajectories: pre-state -> one oracle step == recorded post-state within TOL."""
    N = LINEAR_SUITES[name][0]
    prm = params(oracle, name)
    for case, steps in load_golden('traj_' + name)['trajectories'].items():
        st = fill_host_state(oracle, [s['pre'] for s in steps], N)
        st.g_time[:] = [float(s['global_time']) - 0.25 for s in steps]
        io = oracle.HostStepIO(len(steps))
        io.action[:] = [[float(x) for x in s['action']] for s in steps]
        lin.step(prm, st, io)
        for e, s in enumerate(steps):
            r, h = scene_arrays(s['post'], N)
            assert np.abs(io.action_out[e] - [float(x) for x in s['action']]).max() <= TOL, (case, e)
            assert abs(io.reward[e] - float(s['reward'])) <= TOL and io.done[e] == s['done'] and io.info[e] == s['info']
            if s['dmin'] is not None:
                assert abs(io.dmin[e] - float(s['dmin'])) <= TOL
            assert np.abs(st.r_pos[e] - r[0:2]).max() <= TOL
            assert np.abs(st.h_pos[e] - h[:, 0:2]).max() <= TOL and np.abs(st.h_vel[e] - h[:, 2:4]).max() <= TOL, (case, e)


def test_visible_robot_changes_nothing_for_linear_humans():
    """Linear humans ignore their observation, so the robot's visibility changes no episode of the reference's."""
    a = load_golden('suite_circle5_linear_humans_invisible')
    b = load_golden('suite_circle5_linear_humans_visible')
    assert a['log_lines'] == b['log_lines']
    for x, y in zip(a['cases'], b['cases']):
        assert (x['info'], x['steps'], x['final']['humans'], x['return']) == (y['info'], y['steps'], y['final']['humans'], y['return'])


def test_static_humans_oscillate_and_parked_slots_stay(oracle):
    """Rule `mixed`: a real static human (goal = position, crowd_sim.py:141) steps +x at v_pref (np.arctan2(0, 0) = 0) and
    back (atan2(0, -0.25) = pi), like the reference's; a PARKED slot of the fixed-N layout never moves."""
    from crowdnav_b200 import _abi
    st = oracle.HostState(1, 3)
    st.r_pos[0] = (0.0, -4.0); st.r_goal[0] = (0.0, 4.0); st.r_attr[0] = (0.3, 1.0)
    st.h_pos[0, 0] = st.h_goal[0, 0] = (1.5, 2.0)
    st.h_pos[0, 1] = st.h_goal[0, 1] = (0.0, -10.0)                       # the 0-human dummy of crowd_sim.py:123
    st.h_pos[0, 2] = st.h_goal[0, 2] = (_abi.PARKED_X + 200.0, _abi.PARKED_X)
    st.h_attr[0] = (0.3, 1.0)
    prm, io = oracle.default_params(human_policy=_abi.HUMANS_LINEAR), oracle.HostStepIO(1)
    lin.step(prm, st, io)
    assert tuple(st.h_pos[0, 0]) == (1.5 + 0.25, 2.0) and tuple(st.h_vel[0, 0]) == (1.0, 0.0)
    assert tuple(st.h_pos[0, 1]) == (0.25, -10.0)
    lin.step(prm, st, io)
    assert st.h_vel[0, 0, 0] == -1.0 and st.h_vel[0, 0, 1] == np.sin(np.pi)
    assert st.h_pos[0, 0, 0] == 1.75 - 0.25
    assert tuple(st.h_pos[0, 2]) == (_abi.PARKED_X + 200.0, _abi.PARKED_X) and tuple(st.h_vel[0, 2]) == (0.0, 0.0)


def test_linear_decisions_fixture_has_linear_humans():
    """The SARL / CADRL decisions among linear humans were taken on scenes whose humans walk straight to their goals."""
    d = load_golden('policy_decisions_linear_humans')
    for key in ('cadrl', 'sarl'):
        rows = d[key]['decisions']
        assert len(rows) == 9 and all(len(r['values']) == 81 for r in rows)
        for r in rows:
            if r['step'] == 0:
                continue
            for h in r['scene']['humans']:
                _, _, vx, vy, _, _, _, vp = (float(x) for x in h)
                assert abs(np.hypot(vx, vy) - vp) < 1e-12          # ORCA humans would slow down near each other


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason='needs the reference implementation')
def test_gen_golden_reproduces_linear_fixtures(tmp_path):
    """tests/gen_linear_golden.py, run again from the reference, writes the committed fixtures' content."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'gen_linear_golden.py'), '--out', str(tmp_path)],
                         capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-2000:]
    names = sorted(os.listdir(tmp_path))
    assert len(names) == 13
    for n in names:
        with gzip.open(os.path.join(tmp_path, n), 'rt') as f:
            assert json.load(f) == load_golden(n[:-len('.json.gz')]), n
