"""GPU tests of the Linear policy (env.config [humans] policy = linear; test.py --policy linear) in every kernel that advances
or predicts humans. Bars: CUDA against CUDA bit-identical (flat / crowd / generic kernels, step_n against single steps,
onestep_lookahead against step); CUDA against the oracle and the reference's fixtures within TOL (CUDA's double atan2 is not
glibc's, numpy's scalar arctan2 is neither), terminal classes and step counts identical, float32 rows at 1e-5."""
import logging

import numpy as np
import pytest
import torch

import linear_oracle as lin
from linear_suites import LINEAR_SUITES, TOL
from util import load_golden, scene_arrays, fill_host_state

pytestmark = pytest.mark.gpu

FIELDS = ('h_pos', 'h_vel', 'h_goal', 'h_attr', 'r_pos', 'r_vel', 'r_goal', 'r_attr', 'g_time')
ROBOT = {'orca': 1, 'linear': 3, 'external_xy': 0, 'external_rot': 2}


@pytest.fixture(autouse=True)
def _default_kernel_routing():
    from crowdnav_b200 import _abi, build
    build.build()
    _abi.load().crowdsim_debug_force_generic(0)
    yield
    _abi.load().crowdsim_debug_force_generic(0)


def make_env(B, N, robot_policy, human_policy='linear', rule='circle_crossing', robot_visible=False):
    from crowdnav_b200.batched import BatchedCrowdSim, default_config
    env = BatchedCrowdSim(B)
    env.configure(default_config(human_num=N, test_sim=rule, robot_visible=robot_visible, human_policy=human_policy))
    env.set_robot_policy(robot_policy)
    return env


def random_host(oracle, B, N, seed, parked=False):
    rng = np.random.RandomState(seed)
    st = oracle.HostState(B, N)
    st.h_pos[...] = rng.uniform(-4.5, 4.5, (B, N, 2)); st.h_goal[...] = rng.uniform(-4.5, 4.5, (B, N, 2))
    st.h_vel[...] = rng.uniform(-1, 1, (B, N, 2))
    st.h_attr[..., 0] = rng.uniform(0.2, 0.5, (B, N)); st.h_attr[..., 1] = rng.uniform(0.5, 1.5, (B, N))
    st.r_pos[...] = rng.uniform(-4.5, 4.5, (B, 2)); st.r_vel[...] = rng.uniform(-1, 1, (B, 2)).astype(np.float32)
    st.r_goal[...] = rng.uniform(-4.5, 4.5, (B, 2))
    st.r_attr[:, 0] = rng.uniform(0.2, 0.5, B); st.r_attr[:, 1] = rng.uniform(0.5, 1.5, B)
    st.r_theta[...] = rng.uniform(0, 2 * np.pi, B); st.g_time[...] = 0.25 * rng.randint(0, 99, B)
    if N:
        st.h_goal[::7, 0] = st.h_pos[::7, 0]                 # static humans (rule `mixed`, crowd_sim.py:141)
    if parked and N > 1:
        for e in range(0, B, 3):                             # parked slots of rule `mixed` (crowdsim_b200.h)
            x = 1.0e6 + 100.0 * (N - 1)
            st.h_pos[e, N - 1] = st.h_goal[e, N - 1] = (x, 1.0e6); st.h_vel[e, N - 1] = 0.0
    return st


def assert_close(env, host, io, what):
    dev = env.state.to_host()
    for f in FIELDS:
        d = np.abs(dev[f] - getattr(host, f))
        assert d.max(initial=0.0) <= TOL, '%s: %s max abs %.3g' % (what, f, d.max())
    assert np.array_equal(env.info.cpu().numpy(), io.info) and np.array_equal(env.done.cpu().numpy(), io.done), what
    assert np.abs(env.reward.cpu().numpy() - io.reward).max() <= TOL, what
    live = np.isfinite(io.dmin)
    assert np.abs(env.dmin.cpu().numpy()[live] - io.dmin[live]).max(initial=0.0) <= TOL, what


COMBOS = [('orca', 'linear'), ('linear', 'orca'), ('linear', 'linear'), ('external_xy', 'linear'), ('external_rot', 'linear')]


@pytest.mark.parametrize('N', [1, 5, 10, 20])
@pytest.mark.parametrize('robot,humans', COMBOS)
def test_step_against_oracle(oracle, N, robot, humans):
    """Random scenes (static humans, parked slots), 6 steps; the small-crowd kernel (N <= 5) or the crowd kernel (N > 5)
    against the oracle within TOL, states resynchronised after every step so that differences cannot accumulate."""
    B = 1200
    host = random_host(oracle, B, N, seed=40 + N, parked=True)
    env = make_env(B, N, robot, humans)
    env.state.load_host(host)
    prm = oracle.default_params(robot_policy=ROBOT[robot], human_policy=1 if humans == 'linear' else 0)
    io = oracle.HostStepIO(B)
    rng = np.random.RandomState(3)
    for t in range(6):
        io.action[...] = rng.uniform(0, 1, (B, 2)) if robot == 'external_rot' else rng.uniform(-1, 1, (B, 2))
        env.step(None if robot in ('orca', 'linear') else torch.from_numpy(io.action).to(env.device))
        lin.step(prm, host, io)
        torch.cuda.synchronize()
        assert_close(env, host, io, '%s/%s N=%d step %d' % (robot, humans, N, t))
        if N > 1:
            parked = host.h_pos[::3, N - 1]
            assert np.array_equal(env.state.h_pos[::3, N - 1].cpu().numpy(), parked) and (parked[:, 0] == 1.0e6 + 100.0 * (N - 1)).all()
        env.state.load_host(host)


@pytest.mark.parametrize('N', [1, 5, 10, 20])
@pytest.mark.parametrize('robot,humans', COMBOS[:3])
def test_kernels_and_step_n_bit_identical(oracle, N, robot, humans):
    """The same scenes through (a) the default kernels one step per call, (b) the generic kernel, (c) crowdsim_step_n(8)
    (one launch at N <= 5): every state and output array identical after 8 steps."""
    from crowdnav_b200 import _abi
    B = 900
    host = random_host(oracle, B, N, seed=70 + N, parked=True)
    out = []
    for mode in ('single', 'generic', 'step_n'):
        env = make_env(B, N, robot, humans)
        env.state.load_host(host)
        _abi.load().crowdsim_debug_force_generic(1 if mode == 'generic' else 0)
        n0 = _abi.load().crowdsim_launch_count()
        if mode == 'step_n':
            env.step_n(8)
            if 1 <= N <= 5:
                assert _abi.load().crowdsim_launch_count() - n0 == 1          # one launch, like an ORCA robot
        else:
            for _ in range(8):
                env.step()
        torch.cuda.synchronize()
        out.append((env.state.to_host(), env.reward.cpu().numpy(), env.info.cpu().numpy(), env.action_out.cpu().numpy()))
    _abi.load().crowdsim_debug_force_generic(0)
    for o in out[1:]:
        for f in FIELDS:
            assert np.array_equal(o[0][f], out[0][0][f]), f
        assert np.array_equal(o[1], out[0][1]) and np.array_equal(o[2], out[0][2]) and np.array_equal(o[3], out[0][3])


@pytest.mark.parametrize('N', [1, 5])
@pytest.mark.parametrize('robot,humans', COMBOS[:3])
def test_step_n_equals_single_steps_through_autoreset(N, robot, humans):
    """crowdsim_step_n(n) == n x crowdsim_step through episode ends: auto-reset installs of prefetched scenes and the slot
    accumulators. (Per-slot seeds advanced by B: which slot draws which case from a shared case queue is not deterministic.)"""
    B = 256
    outs = []
    for n in (1, 8):
        env = make_env(B, N, robot, humans)
        ep = env.track_episodes(1)
        env.enable_autoreset('circle_crossing', seed_stride=B)
        env.reset_seeds(np.arange(1000, 1000 + B), rule='circle_crossing', seed_stride=B)
        for it in range(48 // n * 4):
            if it % (8 // n) == 0:
                env.prefetch()
            env.step(n_steps=n)
        torch.cuda.synchronize()
        outs.append((env.state.to_host(), {k: getattr(ep, k).cpu().numpy() for k in ('ep_steps', 'ep_return', 'ep_too_close')},
                     env._seed32.cpu().numpy()))
    for f in FIELDS + ('active',):
        assert np.array_equal(outs[0][0][f], outs[1][0][f]), f
    for k in outs[0][1]:
        assert np.array_equal(outs[0][1][k], outs[1][1][k]), k
    assert np.array_equal(outs[0][2], outs[1][2])
    assert ((outs[0][2].astype(np.int64) - np.arange(1000, 1000 + B)) // B >= 3).sum() > B // 2     # >= 2 installs per slot


@pytest.mark.parametrize('N', [1, 5, 10, 20])
@pytest.mark.parametrize('robot,humans', [('orca', 'linear'), ('linear', 'linear'), ('external_xy', 'linear')])
def test_onestep_lookahead_and_lookahead_humans(oracle, N, robot, humans):
    """crowdsim_onestep_lookahead == the non-mutating part of crowdsim_step (bit-identical); crowdsim_lookahead_humans
    against the oracle within TOL."""
    B = 700
    host = random_host(oracle, B, N, seed=90 + N, parked=True)
    env = make_env(B, N, robot, humans)
    env.state.load_host(host)
    act = torch.from_numpy(np.random.RandomState(1).uniform(-1, 1, (B, 2))).to(env.device)
    (lp, lv, _), r, d, i = env.onestep_lookahead(act)
    lp, lv, r, d, i = lp.cpu().numpy(), lv.cpu().numpy(), r.cpu().numpy().copy(), d.cpu().numpy().copy(), i.cpu().numpy().copy()
    before = env.state.to_host()
    for f in FIELDS:
        assert np.array_equal(before[f], getattr(host, f)), f                 # nothing mutated
    hp, hv = env.lookahead_humans()
    env.step(None if robot != 'external_xy' else act)
    torch.cuda.synchronize()
    after = env.state.to_host()
    assert np.array_equal(lp, after['h_pos']) and np.array_equal(lv, after['h_vel'])
    assert np.array_equal(hp.cpu().numpy(), after['h_pos']) and np.array_equal(hv.cpu().numpy(), after['h_vel'])
    assert np.array_equal(r, env.reward.cpu().numpy()) and np.array_equal(i, env.info.cpu().numpy())
    o_pos, o_vel = lin.lookahead_humans(oracle.default_params(robot_policy=0, human_policy=1), host)
    assert np.abs(hp.cpu().numpy() - o_pos).max() <= TOL and np.abs(hv.cpu().numpy() - o_vel).max() <= TOL


@pytest.mark.parametrize('N', [1, 5, 10, 20])
def test_lookahead_pack_against_oracle(oracle, N):
    """crowdsim_lookahead_pack with linear humans: the N human predictions are N Linear velocities (float64)."""
    B = 300
    host = random_host(oracle, B, N, seed=120 + N)        # (a parked human's float32 rows are ~1e6: no absolute 1e-5 bar)
    env = make_env(B, N, 'external_xy', 'linear')
    env.state.load_host(host)
    from crowdnav_b200.policy import make_sarl
    actions = make_sarl(seed=0).action_space_np
    states, reward = env.lookahead_pack(torch.from_numpy(actions).to(env.device))
    o_states, o_reward = lin.lookahead_pack(oracle.default_params(robot_policy=0, human_policy=1), host, actions)
    assert np.abs(reward.cpu().numpy() - o_reward).max() <= TOL
    assert np.abs(states.cpu().numpy() - o_states).max() < 1e-5


def test_sarl_decisions_among_linear_humans_match_reference(oracle):
    """The reference's SARL (seed-0 weights) among linear humans: per-action values and greedy actions
    (tests/golden/policy_decisions_linear_humans) through lookahead_pack on device."""
    from crowdnav_b200.policy import make_sarl
    d = load_golden('policy_decisions_linear_humans')['sarl']
    rows = d['decisions']
    host = fill_host_state(oracle, [r['scene'] for r in rows], 5)
    host.g_time[:] = [float(r['global_time']) for r in rows]
    env = make_env(len(rows), 5, 'external_xy', 'linear')
    env.state.load_host(host)
    pol = make_sarl(gamma=d['gamma'], seed=d['seed'])
    pol.set_device(env.device)
    act = pol.act_batch(env).cpu().numpy()
    vals = pol.action_values.cpu().numpy()
    for e, r in enumerate(rows):
        ref = np.array([float(v) for v in r['values']])
        assert np.abs(vals[e] - ref).max() < 1e-4, e
        top2 = np.sort(ref)[-2:]
        if top2[1] - top2[0] > 1e-3:
            assert [float(x) for x in r['action']] == [float(x) for x in act[e]], e


@pytest.mark.parametrize('name', sorted(LINEAR_SUITES))
def test_trajectories_against_reference(oracle, name):
    """Each recorded reference step, pre-state -> one CUDA step -> recorded post-state within TOL."""
    N, rule, vis, robot, humans = LINEAR_SUITES[name]
    for case, steps in load_golden('traj_' + name)['trajectories'].items():
        host = fill_host_state(oracle, [s['pre'] for s in steps], N)
        host.g_time[:] = [float(s['global_time']) - 0.25 for s in steps]
        env = make_env(len(steps), N, robot, humans, rule, bool(vis))
        env.state.load_host(host)
        env.step()
        torch.cuda.synchronize()
        dev = env.state.to_host()
        for e, s in enumerate(steps):
            r, h = scene_arrays(s['post'], N)
            assert np.abs(env.action_out[e].cpu().numpy() - [float(x) for x in s['action']]).max() <= TOL
            assert abs(float(env.reward[e]) - float(s['reward'])) <= TOL and int(env.info[e]) == s['info'], (name, case, e)
            assert np.abs(dev['r_pos'][e] - r[0:2]).max() <= TOL and np.abs(dev['h_pos'][e] - h[:, 0:2]).max() <= TOL
            assert np.abs(dev['h_vel'][e] - h[:, 2:4]).max() <= TOL, (name, case, e)


@pytest.mark.parametrize('name,slots', [('circle5_linear_humans_invisible', 128), ('circle5_linear_humans_visible', 500),
                                        ('circle5_linear_robot', 200), ('circle5_linear_both', 64),
                                        ('square20_linear_humans', 32)])
def test_explorer_reproduces_reference(name, slots):
    """BatchedExplorer(env, 'orca' | 'linear') over `slots` env slots: the reference Explorer's log lines, its env-step
    total, and per case the terminal class, steps and (within TOL) the discounted return."""
    from crowdnav_b200.explorer import BatchedExplorer
    N, rule, vis, robot, humans = LINEAR_SUITES[name]
    d = load_golden('suite_' + name)
    k = len(d['cases'])
    env = make_env(slots, N, robot, humans, rule, bool(vis))
    ex = BatchedExplorer(env, robot, gamma=0.9)
    lines = []
    handler = logging.Handler(); handler.emit = lambda rec: lines.append(rec.getMessage())
    root = logging.getLogger(); root.addHandler(handler); old = root.level; root.setLevel(logging.INFO)
    try:
        st = ex.run_k_episodes(k, 'test', print_failure=True)
    finally:
        root.removeHandler(handler); root.setLevel(old)
    assert lines == d['log_lines']
    assert st['env_steps'] == d['total_env_steps']
    rows = ex.last_rows.cpu().numpy()
    for i, c in enumerate(d['cases']):
        assert (int(rows[i, 0]), int(rows[i, 1])) == (c['info'], c['steps']), c['case']
        assert abs(rows[i, 3] - float(c['return'])) <= TOL


def test_mixed_suite_and_static_humans(oracle):
    """Rule `mixed` with linear humans, scenes generated on device: every case's terminal class and step count as in the
    reference; static humans (and the 0-human dummy at (0, -10)) oscillate about their spot, parked slots never move."""
    N = 5
    d = load_golden('suite_mixed5_linear_humans')
    cases = d['cases']
    B = len(cases)
    env = make_env(B, N, 'orca', 'linear', 'mixed')
    ep = env.track_episodes(B)
    host = oracle.HostState(B, N)
    oracle.reset(host, [1000 + c['case'] for c in cases], 'mixed')      # (device generation: test_cuda_0_parity)
    env.state.load_host(host)
    env.episodes.ep_case.copy_(torch.arange(B, dtype=torch.int32))
    start = env.state.to_host()
    env.step()
    torch.cuda.synchronize()
    one = env.state.to_host()
    parked = start['h_pos'][:, :, 0] >= 5.0e5
    static = (start['h_pos'] == start['h_goal']).all(axis=2) & ~parked
    assert parked.any() and static.any()
    assert np.array_equal(one['h_pos'][parked], start['h_pos'][parked])
    assert np.array_equal(one['h_vel'][static], np.tile([[1.0, 0.0]], (int(static.sum()), 1)) * start['h_attr'][static][:, 1:2])
    for _ in range(110):
        env.step()
    torch.cuda.synchronize()
    end = env.state.to_host()
    assert np.array_equal(end['h_pos'][parked], start['h_pos'][parked])
    # A static scene's humans oscillate about their goals, and after a few steps the direction they take is that of a vector of
    # a few ulps: there CUDA's double atan2 and glibc's / numpy's differ by 1 ulp, a velocity's float32 cast differs and the
    # robot's ORCA decision follows it. Case 159 (DESIGN.md §8): step 4, human 2 at (-2.8e-17, 0.25) from its goal,
    # atan2 = pi/2 on the GPU and pi/2 + 1 ulp in the reference; vx 6.1e-17 vs -1.6e-16; collision at step 11 instead of 13.
    # Those cases are findings, not tolerances: every other case must match.
    flips = []
    for i, c in enumerate(cases):
        if (int(ep.res_info[i]), int(ep.res_steps[i])) != (c['info'], c['steps']):
            flips.append(c['case'])
            assert static[i].any() and (static[i] | parked[i]).all(), c['case']
            continue
        assert abs(float(ep.res_return[i]) - float(c['return'])) <= TOL, c['case']
    print('mixed cases that flip on the GPU (static scenes):', flips)
    assert flips == [159]


def test_compat_env_replays_reference_trajectories():
    """gym.make('CrowdSim-v0') with [humans] policy = linear: the reference's test.py flow with an ORCA robot replays the
    recorded trajectory steps of the fixtures (actions, rewards, infos, positions within TOL)."""
    import crowdnav_b200.compat as compat
    from crowdnav_b200.batched import default_config
    compat.install()
    import gym
    from crowd_sim.envs.utils.robot import Robot
    from crowd_sim.envs.policy.orca import ORCA
    from crowd_sim.envs.policy.linear import Linear
    for name, make_policy in (('circle5_linear_humans_invisible', ORCA), ('circle5_linear_both', Linear)):
        cfg = default_config(human_num=5, human_policy='linear')
        env = gym.make('CrowdSim-v0')
        env.configure(cfg)
        robot = Robot(cfg, 'robot')
        policy = make_policy()
        robot.set_policy(policy)
        env.set_robot(robot)
        policy.set_phase('test'); policy.set_device(torch.device('cuda:0')); policy.set_env(env)
        for case, steps in load_golden('traj_' + name)['trajectories'].items():
            ob = env.reset('test', int(case))
            assert type(env.humans[0].policy).__name__ == 'Linear'
            for s in steps:
                action = robot.act(ob)
                ob, reward, done, info = env.step(action)
                r, h = scene_arrays(s['post'])
                assert abs(action.vx - float(s['action'][0])) < 1e-6 and abs(action.vy - float(s['action'][1])) < 1e-6
                assert abs(reward - float(s['reward'])) <= TOL and done == s['done']
                assert abs(robot.px - r[0]) < 1e-6 and abs(robot.py - r[1]) < 1e-6
                assert max(abs(o.px - hh[0]) + abs(o.py - hh[1]) for o, hh in zip(ob, h)) < 1e-9
            assert done
