"""GPU parity away from the default configuration. Every other parity test runs env.config's defaults and orca.py's constants,
where the robot's and the humans' ORCA radii are the same float (both safety spaces 0), every x * time_step is exact
(0.25), and the neighbour range and count (10 m, 10) never cut anything off. Here:
  (a) dense random scenes on every kernel route against the CPU oracle, bit for bit, at
        IL    robot safety space 0.15 (train.py's imitation-learning demonstrations)
        SAFE  human safety space 0.05, robot 0.15
        DT    time step 0.1, time limit 30, time horizon 3, shifted rewards and discomfort distance
        NB    neighbour range 2.5 m, at most 3 neighbours;  NB0 / NB1  at most 0 / 1 neighbour
  (b) the reference's own fixtures at these configurations (tests/gen_config_golden.py) on the device;
  (c) imitation learning end to end at the shift configuration against the reference's Explorer.update_memory."""
import logging

import numpy as np
import pytest
import torch

import config_suites as cs
from util import load_golden, scene_arrays, fill_host_state

pytestmark = pytest.mark.gpu

STATE_FIELDS = ('h_pos', 'h_vel', 'h_goal', 'h_attr', 'r_pos', 'r_vel', 'r_goal', 'r_attr', 'r_theta', 'g_time')

MATRIX = {
    # name: (config of tests/config_suites.py, env attributes set after configure)
    'IL': ('default', dict(robot_safety_space=0.15)),
    'SAFE': ('default', dict(human_safety_space=0.05, robot_safety_space=0.15)),
    'DT': ('shift', dict(time_horizon=3.0)),
    'NB': ('default', dict(neighbor_dist=2.5, max_neighbors=3)),
    'NB0': ('default', dict(max_neighbors=0)),
    'NB1': ('default', dict(max_neighbors=1)),
}
CFGS = sorted(MATRIX)


@pytest.fixture(scope='module')
def make_env():
    assert torch.cuda.is_available(), 'gpu-marked test without a GPU'
    from crowdnav_b200 import _abi, build as cuda_build
    cuda_build.build()
    _abi.load()
    from crowdnav_b200.batched import BatchedCrowdSim

    def make(B, N, cfg=None, config='default', test_sim='circle_crossing', robot_visible=False, robot_policy='orca', **attrs):
        if cfg is not None:
            config, over = MATRIX[cfg]
            attrs = dict(over, **attrs)
        env = BatchedCrowdSim(B)
        env.configure(cs.env_config(config, human_num=N, test_sim=test_sim, robot_visible=robot_visible))
        for k, v in attrs.items():
            setattr(env, k, v)
        env.set_robot_policy(robot_policy)
        return env
    return make


@pytest.fixture(autouse=True)
def _default_kernel_routing():
    from crowdnav_b200 import _abi
    _abi.load().crowdsim_debug_force_generic(0)
    yield
    _abi.load().crowdsim_debug_force_generic(0)


def _policy_code(policy):
    from crowdnav_b200 import _abi
    return {'orca': _abi.ROBOT_ORCA, 'external_xy': _abi.ROBOT_EXTERNAL_XY, 'external_rot': _abi.ROBOT_EXTERNAL_ROT}[policy]


def _params(oracle, cfg, vis, policy='orca'):
    config, over = MATRIX[cfg]
    return oracle.default_params(**dict(cs.CONFIGS[config][0], **over), robot_visible=vis, robot_policy=_policy_code(policy))


def _random_host_state(oracle, cfg, B, N, seed, spread=4.5):
    """The dense random scenes of test_cuda_0_parity, with global times spread over the configuration's episode length (so
    that some envs time out)."""
    p = cs.CONFIGS[MATRIX[cfg][0]][0]
    dt, limit = p.get('time_step', 0.25), p.get('time_limit', 25.0)
    rng = np.random.RandomState(seed)
    st = oracle.HostState(B, N)
    st.h_pos[...] = rng.uniform(-spread, spread, (B, N, 2))
    st.h_vel[...] = rng.uniform(-1, 1, (B, N, 2)).astype(np.float32)
    st.h_goal[...] = rng.uniform(-spread, spread, (B, N, 2))
    st.h_attr[..., 0] = rng.uniform(0.2, 0.5, (B, N)); st.h_attr[..., 1] = rng.uniform(0.5, 1.5, (B, N))
    st.r_pos[...] = rng.uniform(-spread, spread, (B, 2)); st.r_vel[...] = rng.uniform(-1, 1, (B, 2)).astype(np.float32)
    st.r_goal[...] = rng.uniform(-spread, spread, (B, 2))
    st.r_attr[:, 0] = rng.uniform(0.2, 0.5, B); st.r_attr[:, 1] = rng.uniform(0.5, 1.5, B)
    st.r_theta[...] = rng.uniform(0, 2 * np.pi, B)
    st.g_time[...] = dt * rng.randint(0, int(limit / dt), B)
    return st


def _assert_state_equal(env, host, what='', fields=STATE_FIELDS):
    dev = env.state.to_host()
    for f in fields:
        a, b = dev[f], getattr(host, f)
        assert np.array_equal(a, b), '%s: field %s differs in %d entries (max abs %.3g)' % (
            what, f, int((a != b).sum()), float(np.abs(a - b).max()))


def _assert_io_equal(env, io, what=''):
    for f in ('done', 'info', 'reward', 'dmin', 'action_out'):
        a, b = getattr(env, f).cpu().numpy(), getattr(io, f)
        assert np.array_equal(a, b), '%s: %s differs in %d entries' % (what, f, int((a != b).sum()))


def _run_steps(make_env, oracle, cfg, B, N, vis, seed, steps=6, policy='orca', generic=0):
    from crowdnav_b200 import _abi
    host = _random_host_state(oracle, cfg, B, N, seed)
    env = make_env(B, N, cfg, robot_visible=bool(vis), robot_policy=policy)
    env.state.load_host(host)
    _abi.load().crowdsim_debug_force_generic(generic)
    prm = _params(oracle, cfg, vis, policy)
    io = oracle.HostStepIO(B)
    rng = np.random.RandomState(seed + 1)
    for t in range(steps):
        act = None
        if policy != 'orca':
            io.action[...] = rng.uniform(-1, 1, (B, 2))
            act = torch.from_numpy(io.action).to(env.device)
        env.step(act)
        oracle.step(prm, host, io)
        torch.cuda.synchronize()
        what = '%s N=%d vis=%d generic=%d step %d' % (cfg, N, vis, generic, t)
        _assert_state_equal(env, host, what)
        _assert_io_equal(env, io, what)
    return host


# ---- (a) dense random scenes, every route ---------------------------------------------------------------------------------

@pytest.mark.parametrize('N,vis', [(1, 1), (2, 0), (3, 1), (4, 0), (5, 0), (5, 1)])
@pytest.mark.parametrize('cfg', CFGS)
def test_small_crowd_step(make_env, oracle, cfg, N, vis):
    """Small-crowd kernel (N <= 5, step_flat.cuh), per-warp linearProgram3 queue; B = 1501 leaves the last warp and the last
    block partial for every N."""
    _run_steps(make_env, oracle, cfg, 1501, N, vis, seed=1000 + N)


@pytest.mark.parametrize('cfg', CFGS)
def test_small_crowd_block_queue(make_env, oracle, cfg):
    """20 000 envs: the block-compacted linearProgram3 queue of the small-crowd kernel."""
    _run_steps(make_env, oracle, cfg, 20000, 5, 1, seed=1100, steps=4)


@pytest.mark.parametrize('cfg', CFGS)
def test_step_n(make_env, oracle, cfg):
    """crowdsim_step_n, several steps in one launch with the state in registers, against n oracle steps."""
    for N, vis in ((5, 1), (3, 0)):
        B = 1501
        host = _random_host_state(oracle, cfg, B, N, seed=1200 + N)
        env = make_env(B, N, cfg, robot_visible=bool(vis))
        env.state.load_host(host)
        prm = _params(oracle, cfg, vis)
        io = oracle.HostStepIO(B)
        for n in (2, 8, 16):
            env.step_n(n)
            for _ in range(n):
                oracle.step(prm, host, io)
            torch.cuda.synchronize()
            what = 'step_n %s N=%d n=%d' % (cfg, N, n)
            _assert_state_equal(env, host, what)
            _assert_io_equal(env, io, what)


@pytest.mark.parametrize('N', [6, 10, 20, 63])
@pytest.mark.parametrize('cfg', CFGS)
def test_crowd_kernel(make_env, oracle, cfg, N):
    """Crowd kernel (N > 5, step_mid.cuh), robot visible at N = 10 and 63."""
    _run_steps(make_env, oracle, cfg, 1000 if N <= 20 else 300, N, int(N in (10, 63)), seed=1300 + N, steps=4)


@pytest.mark.parametrize('N', [5, 20, 63])
@pytest.mark.parametrize('cfg', CFGS)
def test_generic_kernel(make_env, oracle, cfg, N):
    """The generic kernel forced (crowdsim_common.cuh), including its neighbour-insertion branch at many candidates."""
    _run_steps(make_env, oracle, cfg, 600 if N <= 20 else 200, N, 1, seed=1400 + N, steps=4, generic=1)


@pytest.mark.parametrize('N', [1, 2, 3, 4])
@pytest.mark.parametrize('cfg', CFGS)
def test_external_rot_small_crowd(make_env, oracle, cfg, N):
    """Unicycle robot (external_rot) on the small-crowd kernel: everything bit-exact but the robot's position and heading,
    where CUDA's double cos / sin enter (1e-12); the states are resynchronised after every step."""
    B = 1501
    host = _random_host_state(oracle, cfg, B, N, seed=1500 + N)
    env = make_env(B, N, cfg, robot_visible=True, robot_policy='external_rot')
    env.state.load_host(host)
    prm = _params(oracle, cfg, 1, 'external_rot')
    io = oracle.HostStepIO(B)
    rng = np.random.RandomState(5)
    for t in range(5):
        io.action[:, 0] = rng.uniform(0, 1, B); io.action[:, 1] = rng.uniform(-0.8, 0.8, B)
        env.step(torch.from_numpy(io.action).to(env.device))
        oracle.step(prm, host, io)
        torch.cuda.synchronize()
        dev = env.state.to_host()
        for f in ('h_pos', 'h_vel'):
            assert np.array_equal(dev[f], getattr(host, f)), (cfg, N, t, f)
        assert np.abs(dev['r_pos'] - host.r_pos).max() <= 1e-12 and np.abs(dev['r_theta'] - host.r_theta).max() <= 1e-12
        assert np.array_equal(env.info.cpu().numpy(), io.info) and np.array_equal(env.done.cpu().numpy(), io.done)
        assert np.abs(env.reward.cpu().numpy() - io.reward).max() <= 1e-12
        env.state.load_host(host)


@pytest.mark.parametrize('cfg', CFGS)
def test_orca_act(make_env, oracle, cfg):
    """The robot's ORCA decision alone: the one-thread-per-env kernel (N <= 5) and the generic route (N = 20)."""
    for N in (1, 2, 3, 4, 5, 20):
        B = 1001
        host = _random_host_state(oracle, cfg, B, N, seed=1600 + N)
        env = make_env(B, N, cfg, robot_visible=bool(N % 2), robot_policy='external_xy')
        env.state.load_host(host)
        act = env.orca_act().cpu().numpy()
        ref = oracle.orca_act(_params(oracle, cfg, N % 2), host)
        assert np.array_equal(act, ref), (cfg, N, int((act != ref).any(axis=1).sum()))
        _assert_state_equal(env, host, 'orca_act leaves the state alone')


@pytest.mark.parametrize('cfg', CFGS)
def test_onestep_lookahead(make_env, oracle, cfg):
    import copy
    for N in (3, 12):
        B = 700
        host = _random_host_state(oracle, cfg, B, N, seed=1700 + N)
        env = make_env(B, N, cfg, robot_visible=True, robot_policy='external_xy')
        env.state.load_host(host)
        io = oracle.HostStepIO(B)
        io.action[...] = np.random.RandomState(8).uniform(-1, 1, (B, 2))
        (npos, nvel, _), rew, done, info = env.onestep_lookahead(torch.from_numpy(io.action).to(env.device))
        torch.cuda.synchronize()
        _assert_state_equal(env, host, 'lookahead leaves the state alone')
        stepped = copy.deepcopy(host)
        oracle.step(_params(oracle, cfg, 1, 'external_xy'), stepped, io)
        assert np.array_equal(npos.cpu().numpy(), stepped.h_pos) and np.array_equal(nvel.cpu().numpy(), stepped.h_vel), (cfg, N)
        assert np.array_equal(info.cpu().numpy(), io.info) and np.array_equal(done.cpu().numpy(), io.done)
        assert np.array_equal(rew.cpu().numpy(), io.reward) and np.array_equal(env.dmin.cpu().numpy(), io.dmin)


@pytest.mark.parametrize('cfg', CFGS)
def test_lookahead_humans(make_env, oracle, cfg):
    for N, vis in ((2, 1), (5, 0), (5, 1), (20, 1)):
        B = 700
        host = _random_host_state(oracle, cfg, B, N, seed=1800 + N)
        env = make_env(B, N, cfg, robot_visible=bool(vis), robot_policy='external_xy')
        env.state.load_host(host)
        npos, nvel = env.lookahead_humans()
        torch.cuda.synchronize()
        o_pos, o_vel = oracle.lookahead_humans(_params(oracle, cfg, vis, 'external_xy'), host)
        assert np.array_equal(npos.cpu().numpy(), o_pos) and np.array_equal(nvel.cpu().numpy(), o_vel), (cfg, N, vis)
        _assert_state_equal(env, host, 'state untouched')


@pytest.mark.parametrize('cfg', CFGS)
def test_lookahead_pack(make_env, oracle, cfg):
    """81-action lookahead fused with rotate: rewards bit-exact, rotated rows within 1e-5 (float32 atan2f / cosf / sinf)."""
    speeds = [(np.exp((i + 1) / 5.0) - 1) / (np.e - 1) for i in range(5)]
    rots = np.linspace(0, 2 * np.pi, 16, endpoint=False)
    actions = np.array([[0.0, 0.0]] + [[s * np.cos(r), s * np.sin(r)] for r in rots for s in speeds])
    for N, vis in ((5, 0), (12, 1)):
        B = 257
        host = _random_host_state(oracle, cfg, B, N, seed=1900 + N)
        env = make_env(B, N, cfg, robot_visible=bool(vis), robot_policy='external_xy')
        env.state.load_host(host)
        states, reward = env.lookahead_pack(torch.from_numpy(actions).to(env.device))
        o_states, o_reward = oracle.lookahead_pack(_params(oracle, cfg, vis, 'external_xy'), host, actions)
        assert np.array_equal(reward.cpu().numpy(), o_reward), (cfg, N)
        assert np.abs(states.cpu().numpy() - o_states).max() < 1e-5, (cfg, N)


# ---- (b) the reference's fixtures at non-default configurations -------------------------------------------------------------

def _suite_env(make_env, name, B, **kw):
    N, rule, vis, phase, config, safety = cs.CONFIG_SUITES[name]
    return make_env(B, N, config=config, test_sim=rule, robot_visible=bool(vis), robot_safety_space=safety, **kw)


@pytest.mark.parametrize('name', cs.TRAJ_SUITES)
def test_step_reproduces_config_trajectories(make_env, oracle, name):
    """Each recorded reference step (pre-state, action, reward, info, post-state) bit for bit."""
    N = cs.CONFIG_SUITES[name][0]
    for case, steps in load_golden('traj_' + name)['trajectories'].items():
        host = fill_host_state(oracle, [s['pre'] for s in steps], N)
        host.g_time[:] = cs.pre_times(steps)
        env = _suite_env(make_env, name, len(steps))
        env.state.load_host(host)
        env.step()
        torch.cuda.synchronize()
        dev = env.state.to_host()
        for e, s in enumerate(steps):
            r, h = scene_arrays(s['post'], N)
            assert (env.action_out[e].cpu().numpy() == [float(x) for x in s['action']]).all(), (name, case, e)
            assert float(env.reward[e]) == float(s['reward']) and int(env.done[e]) == int(s['done']) and int(env.info[e]) == s['info'], (name, case, e)
            if s['dmin'] is not None:
                assert float(env.dmin[e]) == float(s['dmin'])
            assert dev['g_time'][e] == float(s['global_time'])
            assert (dev['r_pos'][e] == r[0:2]).all() and (dev['h_pos'][e] == h[:, 0:2]).all() and (dev['h_vel'][e] == h[:, 2:4]).all(), (name, case, e)


def _check_result_rows(ep, env, name, cases):
    N = cs.CONFIG_SUITES[name][0]
    info = ep.res_info.cpu().numpy(); steps = ep.res_steps.cpu().numpy(); t = ep.res_time.cpu().numpy()
    ret = ep.res_return.cpu().numpy(); tc = ep.res_too_close.cpu().numpy(); mds = ep.res_min_dist_sum.cpu().numpy()
    frp = ep.res_final_rpos.cpu().numpy(); hp = env.state.h_pos.cpu().numpy()
    for i, c in enumerate(cases):
        assert info[i] == c['info'] and steps[i] == c['steps'], (name, c['case'])
        assert t[i] == (cs.time_limit(name) if c['info'] == 4 else float(c['global_time'])), (name, c['case'])
        assert ret[i] == float(c['return']) and tc[i] == c['too_close'] and mds[i] == float(c['min_dist_sum']), (name, c['case'])
        r, h = scene_arrays(c['final'], N)
        assert (frp[i] == r[:2]).all() and (hp[i] == h[:, :2]).all(), (name, c['case'])


@pytest.mark.parametrize('mode', ['step', 'step_n'])
@pytest.mark.parametrize('name', sorted(cs.CONFIG_SUITES))
def test_config_suites_from_reference_scenes(make_env, oracle, name, mode):
    """Whole episodes from the reference's initial scenes (single steps, or 16 per launch with episode bookkeeping inside the
    launch): every result row bit for bit."""
    d = load_golden('suite_' + name)
    cases = d['cases']
    N = cs.CONFIG_SUITES[name][0]
    env = _suite_env(make_env, name, len(cases))
    ep = env.track_episodes(len(cases), d['gamma'])
    env.state.load_host(fill_host_state(oracle, [c['init'] for c in cases], N))
    ep.ep_case.copy_(torch.arange(len(cases), dtype=torch.int32))
    limit = cs.max_steps(name)
    if mode == 'step':
        for _ in range(limit):
            env.step()
    else:
        for _ in range(limit // 16 + 1):
            env.step_n(16)
    torch.cuda.synchronize()
    assert int(env.state.active.sum()) == 0
    _check_result_rows(ep, env, name, cases)


@pytest.mark.parametrize('name', sorted(cs.CONFIG_SUITES))
def test_config_suites_device_reset(make_env, oracle, name):
    """Scenes generated on device from the case seeds with the configuration's reset arguments: against the oracle's reset
    (cos / sin aside, bit for bit), then whole episodes with flags exact and final robot positions within 1e-5."""
    N, rule, _, phase, _, _ = cs.CONFIG_SUITES[name]
    d = load_golden('suite_' + name)
    cases = d['cases']
    B = len(cases)
    env = _suite_env(make_env, name, B)
    ep = env.track_episodes(B, d['gamma'])
    env.reset(phase, cases=[c['case'] for c in cases])
    torch.cuda.synchronize()
    host = oracle.HostState(B, N)
    oracle.reset(host, cs.seeds(name, cases), rule, **cs.reset_kw(name))
    dev = env.state.to_host()
    for f in ('h_attr', 'r_pos', 'r_goal', 'r_attr', 'r_vel', 'h_vel', 'g_time', 'r_theta'):
        assert np.array_equal(dev[f], getattr(host, f)), f
    for f in ('h_pos', 'h_goal'):
        tol = 0.0 if rule == 'square_crossing' else 1e-14              # |5 cos| + noise: a few ulp of CUDA's cos / sin
        assert np.abs(dev[f] - getattr(host, f)).max() <= tol, f
    ep.ep_case.copy_(torch.arange(B, dtype=torch.int32))
    for _ in range(cs.max_steps(name)):
        env.step()
    torch.cuda.synchronize()
    assert [int(x) for x in ep.res_info.cpu()] == [c['info'] for c in cases]
    assert [int(x) for x in ep.res_steps.cpu()] == [c['steps'] for c in cases]
    fr = np.array([scene_arrays(c['final'])[0][:2] for c in cases])
    assert np.abs(ep.res_final_rpos.cpu().numpy() - fr).max() < 1e-5


@pytest.mark.parametrize('name,slots', [('shift5_circle', 64), ('shift5_square', 48), ('il5_train', 100)])
def test_config_autoreset_pipeline(make_env, name, slots):
    """Scenes prefetched on device from the case queue and installed by the step kernel (crowdsim_autoreset carries the
    shifted circle radius, robot radius and v_pref): terminal class and step count exact, final positions within 1e-5."""
    N, rule, _, phase, _, _ = cs.CONFIG_SUITES[name]
    d = load_golden('suite_' + name)
    cases = d['cases']
    k = len(cases)
    env = _suite_env(make_env, name, slots)
    ep = env.track_episodes(k, d['gamma'])
    env.set_case_queue(0, k, phase)
    env.enable_autoreset(rule)
    env.reset_seeds(rule=rule, use_queue=True)
    side = torch.cuda.Stream()
    for it in range(20000):
        if it % 2 == 0:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                env.prefetch()
        env.step()
        if it % 64 == 63 and int(env.state.active.sum()) == 0 and int(env.autoreset.want.sum()) == 0:
            break
    torch.cuda.synchronize()
    assert int(env.state.active.sum()) == 0
    assert [int(x) for x in ep.res_info.cpu()] == [c['info'] for c in cases]
    assert [int(x) for x in ep.res_steps.cpu()] == [c['steps'] for c in cases]
    fr = np.array([scene_arrays(c['final'])[0][:2] for c in cases])
    assert np.abs(ep.res_final_rpos.cpu().numpy() - fr).max() < 1e-5


@pytest.mark.parametrize('name', sorted(cs.CONFIG_SUITES))
def test_explorer_reproduces_config_log_lines(make_env, name):
    """BatchedExplorer.run_k_episodes(k, phase, print_failure=True) prints the reference Explorer's lines for the same cases."""
    from crowdnav_b200.explorer import BatchedExplorer
    phase = cs.CONFIG_SUITES[name][3]
    d = load_golden('suite_' + name)
    env = _suite_env(make_env, name, 128)
    lines = []
    handler = logging.Handler(); handler.emit = lambda rec: lines.append(rec.getMessage())
    root = logging.getLogger(); root.addHandler(handler); old = root.level; root.setLevel(logging.INFO)
    try:
        st = BatchedExplorer(env, 'orca', gamma=d['gamma']).run_k_episodes(len(d['cases']), phase, print_failure=True)
    finally:
        root.removeHandler(handler); root.setLevel(old)
    assert lines == d['log_lines']
    assert st['env_steps'] == d['total_env_steps']


@pytest.mark.parametrize('fixture,config', [('human_times_shift', 'shift'), ('human_times', 'default')])
@pytest.mark.parametrize('neighbours', ['orca_defaults', 'env_limits'])
def test_human_times_match_reference(make_env, oracle, fixture, config, neighbours):
    """CrowdSim.get_human_times runs its own centralised simulation with neighborDist 10, maxNeighbors 10, timeHorizon 5
    (crowd_sim.py:220) whatever the env's ORCA agents use: bit for bit, also with max_neighbors = 3 and neighbor_dist = 2 set
    on the env."""
    rows = load_golden(fixture)['rows']
    assert len(rows) >= 6
    attrs = dict(max_neighbors=3, neighbor_dist=2.0, time_horizon=3.0) if neighbours == 'env_limits' else {}
    for r in rows:
        N = r['N']
        host = fill_host_state(oracle, [r['scene']], N)
        host.g_time[:] = float(r['global_time'])
        env = make_env(1, N, config=config, robot_visible=r['robot_visible'], **attrs)
        env.state.load_host(host)
        before = torch.tensor([[float(t) for t in r['human_times_before']]], dtype=torch.float64)
        ht, gt, fp = env.human_times(before)
        torch.cuda.synchronize()
        assert ht[0].tolist() == [float(t) for t in r['human_times']], (r['tag'], r['case'])
        assert float(gt[0]) == float(r['global_time_after'])
        want = np.array([[float(x) for x in r['final_robot']]] + [[float(x) for x in h] for h in r['final_humans']])
        assert np.array_equal(fp[0].cpu().numpy(), want), (r['tag'], r['case'])


# ---- (c) imitation learning end to end ---------------------------------------------------------------------------------------

def test_il_update_memory_matches_reference(make_env):
    """train.py's demonstrations at the shift configuration: BatchedExplorer(env, 'orca', memory, gamma).run_k_episodes(k,
    'train', update_memory=True, imitation_learning=True) with the robot's safety space 0.15 (one slot, so episodes finish in
    case order) stores the reference's (state, value) pairs: values bit for bit, rotated states within 2e-5."""
    from crowdnav_b200.explorer import BatchedExplorer
    from crowdnav_b200.memory import DeviceReplayMemory
    d = load_golden('il_update_memory_shift')
    env = make_env(1, 5, config='shift', robot_safety_space=0.15)
    mem = DeviceReplayMemory(8192, 5, env.device)
    BatchedExplorer(env, 'orca', memory=mem, gamma=d['gamma']).run_k_episodes(d['k'], 'train', update_memory=True,
                                                                             imitation_learning=True, check_every=1)
    assert len(mem) == d['pairs'] > 300
    ref_values = torch.tensor([float(v) for v in d['values']], dtype=torch.float32)
    ref_states = torch.tensor([[[float(x) for x in row] for row in st] for st in d['states']], dtype=torch.float32)
    assert torch.equal(mem.values[:len(mem), 0].cpu(), ref_values)
    assert (mem.states[:len(mem)].cpu() - ref_states).abs().max() < 2e-5


def test_compat_explorer_il_matches_reference():
    """The same demonstrations through the single-env surface: the compat Explorer driving the compat ORCA(safety_space = 0.15)
    in the compat CrowdSim stores the reference's pairs."""
    import crowdnav_b200.compat as compat
    from test_cuda_1_rollout import _torch_rotate
    compat.install()
    import gym
    from crowd_sim.envs.utils.robot import Robot
    from crowd_sim.envs.policy.orca import ORCA
    from crowd_nav.utils.explorer import Explorer
    d = load_golden('il_update_memory_shift')

    class ListMemory(list):
        def push(self, item):
            self.append(item)

    class Target(object):                      # MultiHumanRL.transform without occupancy maps
        def transform(self, state):
            return _torch_rotate(torch.cat([torch.Tensor([state.self_state + h]) for h in state.human_states], dim=0))
    cfg = cs.env_config('shift', human_num=5)
    env = gym.make('CrowdSim-v0'); env.configure(cfg)
    robot = Robot(cfg, 'robot'); pol = ORCA(); robot.set_policy(pol); env.set_robot(robot)
    pol.safety_space, pol.multiagent_training = 0.15, True
    pol.set_phase('train'); pol.set_env(env)
    mem = ListMemory()
    Explorer(env, robot, torch.device('cpu'), memory=mem, gamma=d['gamma'], target_policy=Target()).run_k_episodes(
        d['k'], 'train', update_memory=True, imitation_learning=True)
    assert len(mem) == d['pairs']
    assert [float(v) for _, v in mem] == [float(torch.tensor(float(v), dtype=torch.float32)) for v in d['values']]
    ref_states = torch.tensor([[[float(x) for x in row] for row in st] for st in d['states']], dtype=torch.float32)
    assert (torch.stack([s for s, _ in mem]) - ref_states).abs().max() < 2e-5
