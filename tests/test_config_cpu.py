"""CPU tests away from the default configuration (tests/config_suites.py): the C oracle against the reference's own fixtures of
train.py's imitation-learning demonstrations (ORCA robot with safety_space = 0.15, train phase) and of the `shift`
configuration (time step 0.1, every reward / scene / agent constant moved), the regeneration of those fixtures, and the
imitation-learning discount weights of TrajectoryRecorder."""
import gzip
import json
import os
import subprocess
import sys

import pytest

import config_suites as cs
from util import load_golden, scene_arrays, fill_host_state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = '/root/reference'


@pytest.mark.parametrize('name', sorted(cs.CONFIG_SUITES))
def test_oracle_reproduces_config_suites(oracle, name):
    """Every case of the reference's suite, bit for bit: terminal class, steps, time, discounted return, danger count / sum,
    final robot and human positions and velocities; and the initial scenes from the case seeds."""
    N, rule, vis, phase, _, _ = cs.CONFIG_SUITES[name]
    d = load_golden('suite_' + name)
    cases = d['cases']
    ep, st = oracle.run_episodes(cs.params(oracle, name), N, cs.seeds(name, cases), rule, gamma=d['gamma'],
                                 max_steps=cs.max_steps(name), **cs.reset_kw(name))
    for i, c in enumerate(cases):
        assert ep.res_info[i] == c['info'] and ep.res_steps[i] == c['steps'], c['case']
        assert ep.res_time[i] == (cs.time_limit(name) if c['info'] == 4 else float(c['global_time'])), c['case']
        assert ep.res_return[i] == float(c['return']), c['case']
        assert ep.res_too_close[i] == c['too_close'] and ep.res_min_dist_sum[i] == float(c['min_dist_sum']), c['case']
        r, h = scene_arrays(c['final'], N)
        assert (ep.res_final_rpos[i] == r[:2]).all(), c['case']
        assert (st.h_pos[i] == h[:, :2]).all() and (st.h_vel[i] == h[:, 2:4]).all(), c['case']
    init = oracle.HostState(len(cases), N)
    oracle.reset(init, cs.seeds(name, cases), rule, **cs.reset_kw(name))
    for e, c in enumerate(cases):
        r, h = scene_arrays(c['init'], N)
        assert (init.r_pos[e] == r[0:2]).all() and (init.r_goal[e] == r[4:6]).all() and (init.r_attr[e] == r[6:8]).all()
        assert (init.h_pos[e] == h[:, 0:2]).all() and (init.h_goal[e] == h[:, 4:6]).all() and (init.h_attr[e] == h[:, 6:8]).all(), c['case']


def test_config_suites_leave_the_defaults():
    """The fixtures really are off the defaults: the IL robot is an invisible ORCA robot in the train phase; shift episodes run
    past the 128 steps of a default-sized discount table and the scenes have the shifted radii / speeds / circle."""
    il = load_golden('suite_il5_train')
    assert il['phase'] == 'train' and il['config']['safety_space'] == 0.15 and il['log_lines'][0].startswith('TRAIN')
    for name in ('shift5_circle', 'shift5_square', 'shift10_visible'):
        cases = load_golden('suite_' + name)['cases']
        assert max(c['steps'] for c in cases) > 128, name
        r, h = scene_arrays(cases[0]['init'])
        assert tuple(r[6:8]) == (0.35, 0.8) and (h[:, 6] == 0.25).all() and (h[:, 7] == 1.2).all()
        if 'circle' in name:
            assert tuple(r[:2]) == (0.0, -5.0)


@pytest.mark.parametrize('name', cs.TRAJ_SUITES)
def test_oracle_steps_reproduce_config_trajectories(oracle, name):
    """Every recorded step of the reference's trajectories: pre-state -> one oracle step == recorded post-state, bit for bit."""
    N = cs.CONFIG_SUITES[name][0]
    prm = cs.params(oracle, name)
    n = 0
    for case, steps in load_golden('traj_' + name)['trajectories'].items():
        st = fill_host_state(oracle, [s['pre'] for s in steps], N)
        st.g_time[:] = cs.pre_times(steps)
        io = oracle.HostStepIO(len(steps))
        oracle.step(prm, st, io)
        for e, s in enumerate(steps):
            r, h = scene_arrays(s['post'], N)
            assert (io.action_out[e] == [float(x) for x in s['action']]).all(), (case, e)
            assert io.reward[e] == float(s['reward']) and io.done[e] == s['done'] and io.info[e] == s['info'], (case, e)
            if s['dmin'] is not None:
                assert io.dmin[e] == float(s['dmin'])
            assert st.g_time[e] == float(s['global_time'])
            assert (st.r_pos[e] == r[0:2]).all() and (st.h_pos[e] == h[:, 0:2]).all() and (st.h_vel[e] == h[:, 2:4]).all(), (case, e)
            n += 1
    assert n > 100


def test_safety_space_changes_the_il_episodes(oracle):
    """The IL suite is not reproduced with the robot's safety space at 0, nor with it given to the humans instead: the fixture
    pins which agents' ORCA radius the 0.15 m goes to."""
    name = 'il5_train'
    N, rule = cs.CONFIG_SUITES[name][:2]
    cases = load_golden('suite_' + name)['cases'][:100]
    want = [(c['info'], c['steps']) for c in cases]
    for over in (dict(robot_safety_space=0.0), dict(robot_safety_space=0.0, human_safety_space=0.15)):
        ep, _ = oracle.run_episodes(cs.params(oracle, name, **over), N, cs.seeds(name, cases), rule)
        assert list(zip(ep.res_info.tolist(), ep.res_steps.tolist())) != want, over


class _StandInEnv(object):
    """What TrajectoryRecorder reads of an env."""

    def __init__(self, time_step, v_pref, time_limit=25):
        self.B, self.human_num, self.device = 2, 5, 'cpu'
        self.time_limit, self.time_step, self.robot_v_pref = time_limit, time_step, v_pref


@pytest.mark.parametrize('time_step,v_pref', [(0.25, 1.0), (0.1, 0.8), (0.2, 1.2)])
def test_recorder_il_weights_follow_the_reference(time_step, v_pref):
    """Imitation-learning values: W[t][i] = pow(gamma, max(t - i, 0) * time_step * v_pref) exactly as explorer.py:104 evaluates
    it (left to right), and gamma_bar = pow(gamma, time_step * v_pref) (explorer.py:112)."""
    import torch
    from crowdnav_b200.memory import TrajectoryRecorder
    gamma = 0.9
    env = _StandInEnv(time_step, v_pref, time_limit=30)
    rec = TrajectoryRecorder(env, memory=None, gamma=gamma)
    T = rec.T
    want = torch.tensor([[pow(gamma, max(t - i, 0) * time_step * v_pref) * (1 if t >= i else 0) for i in range(T)]
                         for t in range(T)], dtype=torch.float64)
    assert torch.equal(rec.W, want), int((rec.W != want).sum())
    assert rec.gamma_bar == pow(gamma, time_step * v_pref)


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason='needs the reference implementation')
def test_gen_golden_reproduces_config_fixtures(tmp_path):
    """tests/gen_config_golden.py, run again from the reference, writes the committed fixtures' content."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'gen_config_golden.py'), '--out', str(tmp_path)],
                         capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stderr[-2000:]
    names = sorted(os.listdir(tmp_path))
    assert len(names) == 9
    for n in names:
        with gzip.open(os.path.join(tmp_path, n), 'rt') as f:
            assert json.load(f) == load_golden(n[:-len('.json.gz')]), n
