"""CPU tests of the host-side logic: BatchedExplorer's reductions / log lines / sharding / the one collective (gloo,
world_size 2), and the value-network ports (weights, action space, greedy decision) against reference fixtures."""
import os
import sys

import numpy as np
import pytest
import torch

from util import SUITES, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rows_from_golden(cases):
    rows = [[c['info'], c['steps'], 25.0 if c['info'] == 4 else float(c['global_time']), float(c['return']),
             c['too_close'], float(c['min_dist_sum'])] for c in cases]
    return torch.tensor(rows, dtype=torch.float64)


@pytest.mark.parametrize('name', [n for n in sorted(SUITES) if n not in ('circle5_random_attr', 'mixed5_invisible')])
def test_summarize_emits_reference_log_lines(name):
    """explorer.py:74-90: from per-case rows, the exact lines the reference's own Explorer printed for the same cases."""
    from crowdnav_b200.explorer import summarize
    d = load_golden('suite_' + name)
    lines = []
    stats = summarize(_rows_from_golden(d['cases']), len(d['cases']), 'test', 25, 0.25, print_failure=True, log=lines.append)
    assert lines == d['log_lines']
    assert stats['success'] == d['counts']['success'] and stats['collision'] == d['counts']['collision']
    assert stats['env_steps'] == d['total_env_steps']


def test_shard_range_partitions():
    from crowdnav_b200.explorer import shard_range
    for k in (1, 7, 500, 131072, 131075):
        for world in (1, 2, 3, 8):
            spans = [shard_range(k, r, world) for r in range(world)]
            assert spans[0][0] == 0 and sum(n for _, n in spans) == k
            for (s0, n0), (s1, _) in zip(spans, spans[1:]):
                assert s0 + n0 == s1
            assert max(n for _, n in spans) - min(n for _, n in spans) <= 1


def _gloo_worker(rank, world, port, k, out_dir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from crowdnav_b200.explorer import shard_range, gather_results, summarize
    from util import load_golden as lg
    dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    cases = lg('suite_circle5_invisible')['cases'][:k]
    rows = _rows_from_golden(cases)
    start, n = shard_range(k, rank, world)
    full = gather_results(rows[start:start + n].clone(), k, rank, world)
    assert torch.equal(full, rows)
    if rank == 0:
        lines = []
        summarize(full, k, 'test', 25, 0.25, print_failure=True, log=lines.append)
        with open(os.path.join(out_dir, 'lines.txt'), 'w') as f:
            f.write('\n'.join(lines))
    dist.destroy_process_group()


@pytest.mark.parametrize('k', [500, 333])
def test_two_rank_gather_gloo(tmp_path, k):
    """The N > 1 path on CPU: 2 processes, contiguous case shards (uneven for k = 333), one all_gather of the result rows,
    rank 0 prints the same lines as a single process."""
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() + k) % 2000
    mp.spawn(_gloo_worker, args=(2, port, k, str(tmp_path)), nprocs=2, join=True)
    from crowdnav_b200.explorer import summarize
    cases = load_golden('suite_circle5_invisible')['cases'][:k]
    lines = []
    summarize(_rows_from_golden(cases), k, 'test', 25, 0.25, print_failure=True, log=lines.append)
    assert open(os.path.join(str(tmp_path), 'lines.txt')).read().split('\n') == lines


def test_action_space_matches_reference():
    from crowdnav_b200.policy import build_action_space
    d = load_golden('rotate_lookahead')
    ref = np.array([[float(x) for x in a] for a in d['action_space']])
    assert np.array_equal(build_action_space(1.0), ref)
    assert ref.shape == (81, 2)


def test_sarl_network_port_matches_reference_values():
    """Same construction order => same seed-0 initial weights as the reference's ValueNetwork (sarl.py:9-27); values of
    the reference's own rotated lookahead states agree to float32 round-off, and so does the greedy decision."""
    from crowdnav_b200.policy import make_sarl
    d = load_golden('rotate_lookahead')
    pol = make_sarl(gamma=d['gamma'], seed=d['sarl_seed'])
    model = pol.get_model()
    disc = pow(d['gamma'], 0.25 * 1.0)
    worst = 0.0
    for row in d['rows']:
        states = torch.tensor([[[float(v) for v in r] for r in la['rotated']] for la in row['lookahead']], dtype=torch.float32)
        with torch.no_grad():
            v = model(states)[:, 0].double().numpy()
        ref_v = np.array([float(la['value']) for la in row['lookahead']])
        worst = max(worst, float(np.abs(v - ref_v).max()))
        total = np.array([float(la['reward']) for la in row['lookahead']]) + disc * v
        best = int(np.argmax(total))
        top2 = np.sort(total)[-2:]
        if top2[1] - top2[0] > 1e-5:
            assert [float(x) for x in row['lookahead'][best]['action']] == [float(x) for x in row['sarl_action']]
    assert worst < 1e-6


def test_sarl_state_dict_keys_match_reference_layout():
    from crowdnav_b200.policy import SARLValueNetwork, CADRLValueNetwork
    keys = set(SARLValueNetwork().state_dict().keys())
    assert {'mlp1.0.weight', 'mlp1.2.weight', 'mlp2.0.weight', 'mlp2.2.weight', 'attention.0.weight', 'attention.2.weight',
            'attention.4.weight', 'mlp3.0.weight', 'mlp3.6.weight'} <= keys
    assert SARLValueNetwork().mlp1[0].in_features == 13 and SARLValueNetwork().attention[0].in_features == 200
    assert SARLValueNetwork().mlp3[0].in_features == 56
    assert 'value_network.0.weight' in CADRLValueNetwork().state_dict()


def test_compat_types_and_module_aliases():
    """crowdnav_b200.compat.install(): the reference's import paths resolve; value types keep the reference's contract."""
    import crowdnav_b200.compat as compat
    compat.install(force_gym_shim=True)
    import gym
    from crowd_sim.envs.utils.state import FullState, ObservableState, JointState
    from crowd_sim.envs.utils.action import ActionXY, ActionRot
    from crowd_sim.envs.utils.info import Timeout, ReachGoal, Danger, Collision, Nothing
    from crowd_sim.envs.policy.policy_factory import policy_factory
    from crowd_sim.envs.utils.robot import Robot  # noqa: F401
    from crowd_nav.utils.explorer import Explorer, average  # noqa: F401
    fs = FullState(1, 2, 3, 4, 0.3, 5, 6, 1.0, 0.5); ob = ObservableState(7, 8, 9, 10, 0.4)
    assert fs + ob == (1, 2, 3, 4, 0.3, 5, 6, 1.0, 0.5, 7, 8, 9, 10, 0.4)          # state.py:17-18,36-37 -> the 14-tuple
    assert not isinstance(fs, ObservableState) and fs.position == (1, 2) and fs.goal_position == (5, 6) and ob.velocity == (9, 10)
    JointState(fs, [ob])
    with pytest.raises(AssertionError):
        JointState(ob, [ob])
    assert (str(Timeout()), str(ReachGoal()), str(Danger(0.1)), str(Collision()), str(Nothing())) == \
        ('Timeout', 'Reaching goal', 'Too close', 'Collision', '')
    assert Danger(0.05).min_dist == 0.05 and ActionXY(1, 2).vx == 1 and ActionRot(1, 2).r == 2
    assert set(policy_factory) == {'linear', 'orca', 'none'} and policy_factory['none']() is None
    assert average([]) == 0 and average([1, 2]) == 1.5
    assert type(gym.make('CrowdSim-v0')).__name__ == 'CrowdSim'


def test_bench_reference_arm_emits_contract_json():
    """bench.py --impl reference (CPU only): one JSON line with the driver's keys, cpu_baseline and a zero-copy e2e block."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '12', '--warmup', '3',
                          '--envs', '512'], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    assert line['impl'] == 'reference' and line['unit'] == 'env-steps/s' and line['value'] > 0 and line['vs_baseline'] is None
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert 'workload' in line['config'] and 'model' not in line['config']


def test_graft_entry_build_compiles_everything():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()
    from crowdnav_b200 import _abi
    assert os.path.exists(_abi.LIB_PATH)
    assert os.path.exists(os.path.join(ROOT, 'oracle', '_build', 'libcrowdsim_oracle.so'))
    assert os.path.exists(os.path.join(ROOT, 'oracle', '_build', 'librvo2_oracle.so'))


def test_device_replay_memory_ring_semantics():
    """memory.py:4-28: capacity-bounded ring, position wraps, len saturates."""
    from crowdnav_b200.memory import DeviceReplayMemory
    m = DeviceReplayMemory(5, 2, 'cpu')
    m.push_batch(torch.ones(3, 2, 13), torch.tensor([1., 2., 3.]))
    assert len(m) == 3 and m.position == 3 and not m.is_full()
    m.push_batch(2 * torch.ones(4, 2, 13), torch.tensor([4., 5., 6., 7.]))
    assert len(m) == 5 and m.position == 2 and m.is_full()
    assert m.values[:, 0].tolist() == [6., 7., 3., 4., 5.]
    s, v = m[0]
    assert s.shape == (2, 13) and float(v) == 6.0
    m.clear()
    assert len(m) == 0


def test_il_value_accumulation_equals_reference_formula():
    """explorer.py:104-105 value_i = sum_t pow(gamma, max(t-i,0)*dt*v_pref) * r_t * [t >= i], accumulated forward in t
    through the W matrix of TrajectoryRecorder. Same factors, same order; equal to the last ulp or two of float64 (CPython
    >= 3.12 evaluates sum() with Neumaier compensation, a plain running sum can differ in the last bit) and therefore
    identical after the float32 cast the reference applies (torch.Tensor([value]))."""
    gamma, dt, vp, T = 0.9, 0.25, 1.0, 40
    rng = np.random.RandomState(0)
    rewards = [float(x) for x in rng.uniform(-0.05, 0.0, T) * (rng.uniform(size=T) < 0.3)]
    rewards[-1] = 1.0
    ref = [sum([pow(gamma, max(t - i, 0) * dt * vp) * r * (1 if t >= i else 0) for t, r in enumerate(rewards)]) for i in range(T)]
    W = torch.tensor([[pow(gamma, (t - i) * dt * vp) if i <= t else 0.0 for i in range(T)] for t in range(T)], dtype=torch.float64)
    G = torch.zeros(T, dtype=torch.float64)
    for t, r in enumerate(rewards):
        G += W[t] * r
    assert np.abs(G.numpy() - np.array(ref)).max() <= 4e-16
    assert torch.equal(G.float(), torch.tensor(ref, dtype=torch.float64).float())


def test_network_ports_equal_reference_modules():
    """With the same state_dict loaded, the ported networks reproduce the reference modules' outputs exactly: the
    reference's state_dict layout (keys, shapes) and its outputs on a seeded input with seeded weights are recorded in
    tests/golden/network_ports (oracle/gen_golden.py); the ports load the same weights and must give the same float32s."""
    from util import network_port_input, network_port_weights
    from crowdnav_b200.policy import LSTMRLValueNetwork, SARLValueNetwork, CADRLValueNetwork
    d = load_golden('network_ports')
    x = network_port_input()
    ports = {'lstm_rl_v1': LSTMRLValueNetwork(), 'lstm_rl_v2': LSTMRLValueNetwork(mlp1_dims=(150, 100, 100, 50)),
             'sarl': SARLValueNetwork(), 'cadrl': CADRLValueNetwork()}
    assert set(ports) == set(d)
    for name, mine in ports.items():
        ref = d[name]
        keys_shapes = [(k, tuple(s)) for k, s in ref['keys_shapes']]
        assert [(k, tuple(v.shape)) for k, v in mine.state_dict().items()] == keys_shapes, name
        mine.load_state_dict(network_port_weights(keys_shapes, ref['seed']))
        with torch.no_grad():
            got = mine(x[:, 0] if name == 'cadrl' else x)
        want = torch.tensor([[float(v) for v in row] for row in ref['output']], dtype=torch.float32)
        assert torch.equal(got, want), (name, float((got - want).abs().max()))


def test_om_sarl_policy_logic_matches_reference_on_oracle_backed_env(oracle):
    """Host logic of BatchedValuePolicy with with_om (lookahead rows ++ occupancy maps of the next human states, broadcast
    over the 81 actions, value = reward + gamma^(dt v_pref) V) against the reference's own OM-SARL per-action values and
    greedy actions (tests/golden/occupancy_maps: om_sarl, seed-0 weights). The env is an oracle-backed stand-in here
    (CPU test); tests/test_cuda_1_rollout.py runs the same check on the CUDA path."""
    from util import fill_host_state
    from crowdnav_b200.policy import make_sarl
    o = load_golden('occupancy_maps')['om_sarl']
    rows = o['decisions']
    host = fill_host_state(oracle, [r['scene'] for r in rows], 5)
    host.g_time[:] = [float(r['global_time']) for r in rows]
    prm = oracle.default_params(robot_policy=0)

    class State(object):
        r_pos, r_goal, r_attr = torch.from_numpy(host.r_pos), torch.from_numpy(host.r_goal), torch.from_numpy(host.r_attr)

    class Env(object):
        B, human_num, device, state = len(rows), 5, torch.device('cpu'), State()

        def lookahead_pack(self, actions, out_states=None, out_reward=None):
            s, r = oracle.lookahead_pack(prm, host, actions.numpy())
            return torch.from_numpy(s), torch.from_numpy(r)

        def lookahead_humans(self):
            p, v = oracle.lookahead_humans(prm, host)
            return torch.from_numpy(p), torch.from_numpy(v)

        def occupancy_maps(self, p, v, cell_num, cell_size, channels):
            return torch.from_numpy(oracle.occupancy_maps(p.numpy(), v.numpy(), cell_num, cell_size, channels))

    pol = make_sarl(gamma=o['gamma'], seed=o['seed'], with_om=True, cell_num=o['cell_num'], cell_size=float(o['cell_size']),
                    om_channel_size=o['om_channel_size'])
    act = pol.act_batch(Env()).numpy()
    vals = pol.action_values.numpy()
    for e, r in enumerate(rows):
        ref = np.array([float(v) for v in r['values']])
        assert np.abs(vals[e] - ref).max() < 1e-5, e
        assert [float(x) for x in r['action']] == [float(x) for x in act[e]], e


def test_compat_agent_kinematics():
    """crowdnav_b200.compat.agents.Agent: agent.py:47-138 semantics (set / accessors / holonomic and unicycle stepping /
    goal test) on hand-computed values. (Bit-exact equivalence with the reference class on thousands of random steps was
    checked in the dev container when the class was written; numpy's cos/sin are used like the reference does.)"""
    from crowdnav_b200.batched import default_config
    from crowdnav_b200.compat.agents import Agent, Robot
    from crowdnav_b200.compat.statetypes import ActionXY, ActionRot
    cfg = default_config()
    a = Agent(cfg, 'humans')
    assert (a.radius, a.v_pref, a.visible, a.sensor, a.kinematics) == (0.3, 1.0, True, 'coordinates', 'holonomic')
    a.time_step = 0.25
    a.set(1.0, 2.0, 5.0, 6.0, 0.1, 0.2, 0.5)
    assert (a.get_position(), a.get_goal_position(), a.get_velocity()) == ((1.0, 2.0), (5.0, 6.0), (0.1, 0.2))
    assert a.compute_position(ActionXY(1.0, -2.0), 0.25) == (1.25, 1.5)
    nxt = a.get_next_observable_state(ActionXY(1.0, -2.0))
    assert (nxt.px, nxt.py, nxt.vx, nxt.vy, nxt.radius) == (1.25, 1.5, 1.0, -2.0, 0.3)
    a.step(ActionXY(1.0, -2.0))
    assert (a.px, a.py, a.vx, a.vy, a.theta) == (1.25, 1.5, 1.0, -2.0, 0.5)
    with pytest.raises(AssertionError):
        a.step(ActionRot(1.0, 0.0))
    a.set(1, 2, 1.1, 2.1, 0, 0, 0, radius=0.4, v_pref=1.3)
    assert (a.radius, a.v_pref) == (0.4, 1.3) and a.reached_destination()
    a.set(1, 2, 2, 3, 0, 0, 0)
    assert not a.reached_destination()
    a.set_position((3, 4)); a.set_velocity([5, 6])
    assert (a.px, a.py, a.vx, a.vy) == (3, 4, 5, 6)
    u = Agent(cfg, 'humans'); u.kinematics = 'unicycle'; u.time_step = 0.25
    u.set(0.0, 0.0, 1.0, 1.0, 0.0, 0.0, np.pi / 2)
    u.step(ActionRot(1.0, np.pi / 2))                       # turn left by 90 degrees, then 0.25 m along -x
    assert abs(u.px + 0.25) < 1e-15 and abs(u.py) < 1e-15 and abs(u.theta - np.pi) < 1e-15
    assert abs(u.vx + 1.0) < 1e-15 and abs(u.vy) < 1e-15
    r = Robot(cfg, 'robot')
    assert r.policy is None and r.visible is False
    with pytest.raises(AttributeError):
        r.act([])


def test_compat_explorer_on_scripted_env():
    """crowdnav_b200.compat.explorer.Explorer (explorer.py:21-125 surface) on a scripted environment: log lines equal
    the shared reducer's on the same episodes, discounted returns / IL values / RL bootstraps follow the reference's
    formulas (exponent (t * time_step) * v_pref), timeouts are not stored, bad end signals raise."""
    import logging
    from crowdnav_b200.compat.explorer import Explorer
    from crowdnav_b200.compat.statetypes import Collision, Danger, Nothing, ReachGoal, Timeout
    from crowdnav_b200.explorer import summarize

    script = [  # per episode: list of (reward, info) ; the last step ends the episode
        [(0.0, Nothing()), (-0.02, Danger(0.12)), (1.0, ReachGoal())],
        [(-0.01, Danger(0.18)), (-0.25, Collision())],
        [(0.0, Nothing())] * 3 + [(0.0, Timeout())],
    ]

    class Policy(object):
        last_state = None

        def set_phase(self, phase):
            self.phase = phase

        def transform(self, state):
            return state * 2

    from crowdnav_b200.batched import default_config
    from crowdnav_b200.compat.agents import Robot as CompatRobot

    class Robot(CompatRobot):
        # the REAL compat Robot: time_step is None until env.reset() assigns it (agent.py:36, crowd_sim.py:296-298) -- a
        # fake with a class-level time_step once hid a read-before-reset bug in run_k_episodes from the CPU suite
        def act(self, ob):
            self.policy.last_state = torch.tensor([float(ob)])
            return ob

    class Env(object):
        time_limit = 25
        global_time = 0.0

        def __init__(self, robot=None):
            self.ep = -1; self.robot = robot

        def reset(self, phase):
            self.ep += 1; self.t = 0; self.global_time = 0.0
            if self.robot is not None:
                self.robot.time_step = 0.25               # like CrowdSim.reset (crowd_sim.py:296-298)
            return 100 * self.ep

        def step(self, action):
            r, info = script[self.ep][self.t]
            self.t += 1; self.global_time += 0.25
            return 100 * self.ep + self.t, r, self.t == len(script[self.ep]), info

    class Memory(list):
        def push(self, item):
            self.append(item)

    lines = []
    handler = logging.Handler(); handler.emit = lambda rec: lines.append(rec.getMessage())
    root = logging.getLogger(); root.addHandler(handler); old = root.level; root.setLevel(logging.INFO)
    mem = Memory()
    robot = Robot(default_config(), 'robot'); robot.policy = Policy(); robot.v_pref = 1.3
    assert robot.time_step is None
    ex = Explorer(Env(robot), robot, torch.device('cpu'), memory=mem, gamma=0.9, target_policy=robot.policy)
    try:
        ex.run_k_episodes(3, 'val', update_memory=True, imitation_learning=True, episode=7, print_failure=True)
    finally:
        root.removeHandler(handler); root.setLevel(old)
    g = lambda t: pow(0.9, t * 0.25 * 1.3)  # noqa: E731
    rets = [g(1) * -0.02 + g(2) * 1.0, -0.01 + g(1) * -0.25, 0.0]
    rows = torch.tensor([[2, 3, 0.75, rets[0], 1, 0.12], [3, 2, 0.5, rets[1], 1, 0.18], [4, 4, 25, rets[2], 0, 0.0]], dtype=torch.float64)
    expect = []
    summarize(rows, 3, 'val', 25, 0.25, episode=7, print_failure=True, log=expect.append)
    assert lines == expect and 'in episode 7' in lines[0] and lines[-1] == 'Timeout cases: 2'
    # imitation learning: 3 + 2 pairs (the timeout episode is not stored), state transformed, value = return-to-go
    assert len(mem) == 5
    assert float(mem[0][0]) == 0.0 and float(mem[1][0]) == 2.0 and float(mem[3][0]) == 200.0
    want = [rets[0], -0.02 + g(1) * 1.0, 1.0, rets[1], -0.25]
    assert [float(v) for _, v in mem] == [float(torch.Tensor([w])) for w in want]
    # RL targets: reward + gamma^(dt v_pref) * V_target(next state); terminal step: the reward
    mem2 = Memory()
    ex2 = Explorer(Env(), robot, torch.device('cpu'), memory=mem2, gamma=0.9)
    ex2.update_target_model(torch.nn.Linear(1, 1))
    with torch.no_grad():
        ex2.target_model.weight.fill_(0.5); ex2.target_model.bias.fill_(0.25)
    ex2.update_memory([torch.tensor([1.0]), torch.tensor([3.0])], None, [0.1, -0.25])
    assert float(mem2[0][1]) == float(torch.Tensor([0.1 + pow(0.9, 0.25 * 1.3) * (0.5 * 3.0 + 0.25)])) and float(mem2[1][1]) == -0.25
    with pytest.raises(ValueError):
        Explorer(Env(), robot, torch.device('cpu')).update_memory([], None, [])
    bad = Env(); script.append([(0.0, Nothing())])
    bad.ep = 2
    with pytest.raises(ValueError):
        Explorer(bad, robot, torch.device('cpu'), gamma=0.9).run_k_episodes(1, 'test')


def _oracle_backed_env(oracle, rows):
    """Stand-in for BatchedCrowdSim in CPU tests of the policy host logic: the kernels' outputs come from the oracle."""
    from util import fill_host_state
    host = fill_host_state(oracle, [r['scene'] for r in rows], 5)
    host.g_time[:] = [float(r['global_time']) for r in rows]
    prm = oracle.default_params(robot_policy=0)

    class State(object):
        r_pos, r_goal, r_attr = torch.from_numpy(host.r_pos), torch.from_numpy(host.r_goal), torch.from_numpy(host.r_attr)

    class Env(object):
        B, human_num, device, state = len(rows), 5, torch.device('cpu'), State()

        def lookahead_pack(self, actions, out_states=None, out_reward=None):
            s, r = oracle.lookahead_pack(prm, host, actions.numpy())
            return torch.from_numpy(s), torch.from_numpy(r)

        def lookahead_humans(self):
            p, v = oracle.lookahead_humans(prm, host)
            return torch.from_numpy(p), torch.from_numpy(v)

        def occupancy_maps(self, p, v, cell_num, cell_size, channels):
            return torch.from_numpy(oracle.occupancy_maps(p.numpy(), v.numpy(), cell_num, cell_size, channels))
    return Env()


def test_epsilon_greedy_and_per_env_discount(oracle):
    """Train-phase predict (multi_human_rl.py:27-31): with probability epsilon a uniformly drawn action of the 81-action
    space, per env; greedy otherwise and always in the val / test phases. The discount of the one-step value uses the
    robot's v_pref of THAT env (multi_human_rl.py:52: pow(gamma, time_step * state.self_state.v_pref))."""
    from crowdnav_b200.policy import make_cadrl
    rows = load_golden('policy_decisions')['cadrl']['decisions'] * 40          # 360 envs
    env = _oracle_backed_env(oracle, rows)
    B = env.B
    pol = make_cadrl(gamma=0.9, seed=0)
    greedy = pol.act_batch(env).clone()
    assert pol.explored is None
    pol.set_phase('train'); pol.set_seed(3)
    pol.set_epsilon(0.0)
    assert torch.equal(pol.act_batch(env), greedy) and pol.explored is None
    pol.set_epsilon(1.0)
    a1 = pol.act_batch(env)
    assert bool(pol.explored.all())
    space = torch.from_numpy(pol.action_space_np)
    assert all(bool((space == a1[e]).all(dim=1).any()) for e in range(B))       # every action is one of the 81
    assert len({tuple(x) for x in a1.tolist()}) > 40                             # drawn per env, not one draw for the batch
    pol.set_epsilon(0.3)
    pol.act_batch(env)
    frac = float(pol.explored.double().mean())
    assert 0.2 < frac < 0.4
    keep = ~pol.explored
    assert torch.equal(pol.act_batch(env)[keep & ~pol.explored], greedy[keep & ~pol.explored])
    pol.set_phase('val')
    assert torch.equal(pol.act_batch(env), greedy) and pol.explored is None
    # per-env v_pref in the discount
    pol.set_phase('test')
    v0 = pol.action_values.clone()
    env.state.r_attr[:, 1] = torch.linspace(0.5, 1.5, B, dtype=torch.float64)
    pol.act_batch(env)
    s, r = env.lookahead_pack(pol.actions)
    vnet = pol.model(s.view(B * 81 * 5, 13)).view(B, 81, 5).min(dim=2).values.double()
    for e in (0, B // 2, B - 1):
        want = r[e] + pow(0.9, 0.25 * float(env.state.r_attr[e, 1])) * vnet[e]
        assert (pol.action_values[e] - want).abs().max() < 1e-12
    assert not torch.allclose(pol.action_values, v0)


@pytest.mark.parametrize('key', ['cadrl', 'lstm_rl', 'lstm_rl_interaction'])
def test_cadrl_and_lstm_rl_policy_logic_matches_reference(oracle, key):
    """BatchedValuePolicy for CADRL (min over the per-human values, cadrl.py:163-166) and LSTM-RL (with query_env the
    lookahead rows reach the LSTM in env order, SURVEY quirk 9) against the reference's own per-action values and greedy
    actions (tests/golden/policy_decisions: seed-0 weights, policy.config defaults)."""
    from crowdnav_b200.policy import make_cadrl, make_lstm_rl
    d = load_golden('policy_decisions')[key]
    rows = d['decisions']
    pol = {'cadrl': lambda: make_cadrl(gamma=d['gamma'], seed=d['seed']),
           'lstm_rl': lambda: make_lstm_rl(gamma=d['gamma'], seed=d['seed']),
           'lstm_rl_interaction': lambda: make_lstm_rl(gamma=d['gamma'], seed=d['seed'], with_interaction_module=True)}[key]()
    act = pol.act_batch(_oracle_backed_env(oracle, rows)).numpy()
    vals = pol.action_values.numpy()
    for e, r in enumerate(rows):
        ref = np.array([float(v) for v in r['values']])
        assert np.abs(vals[e] - ref).max() < 1e-5, (key, e, float(np.abs(vals[e] - ref).max()))
        top2 = np.sort(ref)[-2:]
        if top2[1] - top2[0] > 1e-4:
            assert [float(x) for x in r['action']] == [float(x) for x in act[e]], (key, e)


def test_bench_reference_arm_contract():
    """bench.py --impl reference (the CPU arm run next to ours): one JSON line with the contract's keys, the thread
    calibration bounded by the usable CPUs, a sane rate."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--envs', '256', '--steps', '5', '--warmup', '3',
                          '--no-python-loop'], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-1000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d['impl'] == 'reference' and d['unit'] == 'env-steps/s' and d['higher_is_better'] is True and d['steps'] == 5
    assert d['value'] > 1e5 and d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and 1 <= cb['cores'] <= len(os.sched_getaffinity(0))
    assert str(cb['cores']) in cb['calibration_env_steps_per_s'] and d['gpu_launches'] == 0
