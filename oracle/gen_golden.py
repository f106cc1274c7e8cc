#!/usr/bin/env python
"""Generate tests/golden/*.json.gz by running the REFERENCE'S OWN PYTHON, unmodified, from /root/reference.

TEST INFRASTRUCTURE. Runs only in the build container (the GPU box has no /root/reference); the JSON
fixtures it writes are committed and travel. The reference is imported with three shims on sys.path
(oracle/shims: gym, matplotlib, rvo2); `rvo2` is our float32 restatement of the RVO2 agent step
(oracle/rvo2_sim.c) because the real Python-RVO2 is an absent, unpinned dependency (SURVEY.md 8c).

What is recorded (floats as repr() strings, exact round trip):
  suite_*.json   per test case: terminal info, steps, env.global_time, final robot/human positions,
                 discounted return (explorer.py:71-72), danger count / min_dist sum, plus the log lines the
                 reference's Explorer.run_k_episodes prints for the same cases (explorer.py:80-90)
  traj_*.json    full per-step trajectories of a few cases (every agent position/velocity, reward, info)
  reset_*.json   initial scenes straight after env.reset (scenario generators + MT19937)
  rotate.json    CADRL.rotate + one-step lookahead inputs/outputs of MultiHumanRL.predict's inner loop
  occupancy_maps.json  MultiHumanRL.build_occupancy_maps on scene / lookahead / random human states
  policy_decisions.json  per-action values and greedy actions of the reference's CADRL / LSTM-RL policies
  network_ports.json     outputs of the reference's value-network modules with seeded weights loaded

usage: python oracle/gen_golden.py [--quick]
"""
import configparser
import gzip
import io
import json
import logging
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = '/root/reference'
sys.path.insert(0, os.path.join(HERE, 'shims'))
sys.path.insert(0, REF)
sys.path.insert(0, HERE)

import build as _oracle_build  # noqa: E402

_oracle_build.build()

import numpy as np  # noqa: E402
import torch  # noqa: E402
import gym  # noqa: E402
import crowd_sim  # noqa: E402,F401  (registers CrowdSim-v0)
from crowd_sim.envs.utils.robot import Robot  # noqa: E402
from crowd_sim.envs.utils.info import Timeout, ReachGoal, Danger, Collision, Nothing  # noqa: E402
from crowd_sim.envs.utils.action import ActionXY  # noqa: E402
from crowd_sim.envs.utils.state import JointState  # noqa: E402
from crowd_sim.envs.policy.orca import ORCA  # noqa: E402
from crowd_nav.utils.explorer import Explorer  # noqa: E402
from crowd_nav.policy.policy_factory import policy_factory  # noqa: E402
from crowd_nav.policy import cadrl, lstm_rl, sarl  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, 'tests'))
from util import network_port_input, network_port_weights  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
INFO_CODE = {Nothing: 0, Danger: 1, ReachGoal: 2, Collision: 3, Timeout: 4}


def R(x):
    return repr(float(x))


def make_env(human_num=5, test_sim='circle_crossing', robot_visible=False, randomize=False, policy_name='orca',
             policy_config=None):
    cfg = configparser.RawConfigParser()
    cfg.read(os.path.join(REF, 'crowd_nav', 'configs', 'env.config'))
    cfg.set('sim', 'human_num', str(human_num))
    cfg.set('robot', 'visible', 'true' if robot_visible else 'false')
    cfg.set('env', 'randomize_attributes', 'true' if randomize else 'false')
    env = gym.make('CrowdSim-v0')
    env.configure(cfg)
    env.test_sim = test_sim
    robot = Robot(cfg, 'robot')
    policy = policy_factory[policy_name]()
    if policy_config is not None:
        policy.configure(policy_config)
    else:
        policy.configure(cfg)
    robot.set_policy(policy)
    env.set_robot(robot)
    policy.set_phase('test')
    policy.set_device(torch.device('cpu'))
    policy.set_env(env)
    if isinstance(policy, ORCA):
        policy.safety_space = 0
    return env, robot, cfg


def scene(env):
    r = env.robot
    return {
        'robot': [R(r.px), R(r.py), R(r.vx), R(r.vy), R(r.gx), R(r.gy), R(r.radius), R(r.v_pref), R(r.theta)],
        'humans': [[R(h.px), R(h.py), R(h.vx), R(h.vy), R(h.gx), R(h.gy), R(h.radius), R(h.v_pref)] for h in env.humans],
    }


def run_suite(name, cases, phase='test', gamma=0.9, record_traj=(), fresh_robot_sim=False, reset_human_num=None, **kw):
    """fresh_robot_sim: drop the robot's cached rvo2 sim before every episode. The reference keeps it across
    episodes (orca.py:95-104), so with randomize_attributes the robot would keep solving with the human radii of
    the FIRST episode it saw -- an accident of object lifetime we do not reproduce (DESIGN.md, quirks)."""
    """reset_human_num: rule `mixed` overwrites env.human_num with the drawn count (crowd_sim.py:115) and reset() sizes
    human_times from the STALE value (:263), so the reference's own step() raises IndexError (:404-407) as soon as an
    episode draws more humans than the previous one. The fixture driver therefore restores env.human_num before every
    reset; the reference's Explorer cannot run such a suite at all (no log lines)."""
    env, robot, _ = make_env(**kw)
    # 1) the reference's own Explorer, capturing its log lines
    stream = io.StringIO()
    handler = logging.StreamHandler(stream)
    handler.setFormatter(logging.Formatter('%(message)s'))
    root = logging.getLogger()
    root.addHandler(handler)
    root.setLevel(logging.INFO)
    explorer = Explorer(env, robot, torch.device('cpu'), gamma=gamma)
    env.case_counter[phase] = cases[0]
    if reset_human_num is None:
        explorer.run_k_episodes(len(cases), phase, print_failure=True)
    root.removeHandler(handler)
    log_lines = [l for l in stream.getvalue().splitlines() if l]

    # 2) the same episodes again through reset/act/step, recording per-case details
    env, robot, _ = make_env(**kw)
    per_case = []
    trajs = {}
    total_steps = 0
    for case in cases:
        if fresh_robot_sim:
            robot.policy.sim = None
        if reset_human_num is not None:
            env.human_num = reset_human_num
        ob = env.reset(phase, case)
        init = scene(env)
        done = False
        rewards = []
        too_close = 0
        min_dist_sum = 0.0
        steps = []
        while not done:
            action = robot.act(ob)
            pre = scene(env) if case in record_traj else None
            ob, reward, done, info = env.step(action)
            rewards.append(reward)
            if isinstance(info, Danger):
                too_close += 1
                min_dist_sum += info.min_dist
            if case in record_traj:
                steps.append({'pre': pre, 'action': [R(action.vx), R(action.vy)], 'reward': R(reward),
                              'done': bool(done), 'info': INFO_CODE[type(info)],
                              'dmin': R(info.min_dist) if isinstance(info, Danger) else None,
                              'post': scene(env), 'global_time': R(env.global_time)})
        ret = sum([pow(gamma, t * robot.time_step * robot.v_pref) * r for t, r in enumerate(rewards)])
        total_steps += len(rewards)
        per_case.append({'case': case, 'info': INFO_CODE[type(info)], 'steps': len(rewards),
                         'global_time': R(env.global_time), 'return': R(ret), 'too_close': too_close,
                         'min_dist_sum': R(min_dist_sum), 'final': scene(env), 'init': init})
        if case in record_traj:
            trajs[str(case)] = steps
    counts = {k: sum(1 for c in per_case if c['info'] == v) for k, v in
              (('success', 2), ('collision', 3), ('timeout', 4))}
    if fresh_robot_sim:
        log_lines = []      # Explorer ran with the stale-radius sim; its aggregate lines do not apply
    out = {'name': name, 'phase': phase, 'config': {k: (v if not isinstance(v, bool) else v) for k, v in kw.items()},
           'gamma': gamma, 'log_lines': log_lines, 'counts': counts, 'total_env_steps': total_steps,
           'cases': per_case}
    with gzip.open(os.path.join(OUT, 'suite_%s.json.gz' % name), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))
    if trajs:
        with gzip.open(os.path.join(OUT, 'traj_%s.json.gz' % name), 'wt') as f:
            json.dump({'name': name, 'config': kw, 'trajectories': trajs}, f, separators=(',', ':'))
    print(name, counts, 'env-steps', total_steps)
    for l in log_lines:
        print('   ', l)
    return out


def run_mixed():
    run_suite('mixed5_invisible', list(range(300)), human_num=5, test_sim='mixed', reset_human_num=5, record_traj=(1, 4, 8))


def run_resets():
    """Initial scenes only: scenario generators + MT19937 (crowd_sim.py:155-207, 251-312)."""
    out = {}
    for name, kw, phase, cases in [
        ('circle5_test', dict(human_num=5, test_sim='circle_crossing'), 'test', list(range(0, 40))),
        ('square5_test', dict(human_num=5, test_sim='square_crossing'), 'test', list(range(0, 40))),
        ('square20_test', dict(human_num=20, test_sim='square_crossing'), 'test', list(range(0, 20))),
        ('circle10_test', dict(human_num=10, test_sim='circle_crossing'), 'test', list(range(0, 20))),
        ('circle5_random_attr', dict(human_num=5, test_sim='circle_crossing', randomize=True), 'test', list(range(0, 20))),
        ('square5_random_attr', dict(human_num=5, test_sim='square_crossing', randomize=True), 'test', list(range(0, 20))),
        ('mixed5_test', dict(human_num=5, test_sim='mixed'), 'test', list(range(0, 120))),
        ('mixed5_random_attr', dict(human_num=5, test_sim='mixed', randomize=True), 'test', list(range(0, 40))),
        ('circle5_train', dict(human_num=5, test_sim='circle_crossing'), 'train', [0, 1, 2, 1000, 123456, 4294965294]),
        ('circle5_val', dict(human_num=5, test_sim='circle_crossing'), 'val', [0, 1, 99]),
    ]:
        env, robot, _ = make_env(**kw)
        robot.policy.multiagent_training = True     # ORCA leaves it None; train/val then use human_num (crowd_sim.py:278)
        rows = []
        for c in cases:
            env.reset(phase, c)
            offset = {'train': 2000, 'val': 0, 'test': 1000}[phase]
            rows.append({'case': c, 'seed': offset + c, 'scene': scene(env)})
        out[name] = {'config': kw, 'phase': phase, 'rows': rows}
    with gzip.open(os.path.join(OUT, 'reset_scenes.json.gz'), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))
    print('reset scenes written')


def run_rotate():
    """CADRL.rotate and the inner loop of MultiHumanRL.predict (multi_human_rl.py:35-45), reference code only."""
    pcfg = configparser.RawConfigParser()
    pcfg.read(os.path.join(REF, 'crowd_nav', 'configs', 'policy.config'))
    torch.manual_seed(0)
    env, robot, _ = make_env(human_num=5, test_sim='circle_crossing', policy_name='sarl', policy_config=pcfg)
    policy = robot.policy
    rows = []
    for case in (0, 3, 7):
        ob = env.reset('test', case)
        orca_robot = ORCA()
        orca_robot.time_step = env.time_step
        for step in range(12):
            state = JointState(robot.get_full_state(), ob)
            if policy.action_space is None:
                policy.build_action_space(state.self_state.v_pref)
            if step % 4 == 0:
                per_action = []
                for action in policy.action_space:
                    next_self_state = policy.propagate(state.self_state, action)
                    next_human_states, reward, done, info = env.onestep_lookahead(action)
                    batch = torch.cat([torch.Tensor([next_self_state + nhs]) for nhs in next_human_states], dim=0)
                    rot = policy.rotate(batch)
                    with torch.no_grad():
                        value = policy.model(rot.unsqueeze(0)).data.item()
                    per_action.append({'action': [R(action.vx), R(action.vy)], 'reward': R(reward), 'value': R(value),
                                       'rotated': [[R(v) for v in row] for row in rot.tolist()]})
                cur = torch.cat([torch.Tensor([state.self_state + hs]) for hs in state.human_states], dim=0)
                np_state = np.random.get_state()
                chosen = policy.predict(state)                # the reference's own greedy decision (SARL, seed-0 weights)
                np.random.set_state(np_state)
                rows.append({'case': case, 'step': step, 'scene': scene(env), 'global_time': R(env.global_time),
                             'sarl_action': [R(chosen.vx), R(chosen.vy)],
                             'rotated_current': [[R(v) for v in row] for row in policy.rotate(cur).tolist()],
                             'lookahead': per_action})
            # drive the robot with ORCA so the scene evolves through interesting states
            action = orca_robot.predict(state)
            ob, reward, done, info = env.step(ActionXY(action.vx, action.vy))
            if done:
                break
    space = [[R(a.vx), R(a.vy)] for a in policy.action_space]
    with gzip.open(os.path.join(OUT, 'rotate_lookahead.json.gz'), 'wt') as f:
        json.dump({'action_space': space, 'sarl_seed': 0, 'gamma': policy.gamma, 'rows': rows}, f, separators=(',', ':'))
    print('rotate/lookahead rows', len(rows))


def run_om():
    """MultiHumanRL.build_occupancy_maps (multi_human_rl.py:109-163), reference code only: (a) on the humans of real
    scenes a few steps into test episodes and on the next human states env.onestep_lookahead returns, (b) on random
    dense crowds (N = 3, 8, 20). Stored: inputs (px, py, vx, vy per human) and the reference's float32 maps."""
    from crowd_sim.envs.utils.state import ObservableState
    pcfg = configparser.RawConfigParser()
    pcfg.read(os.path.join(REF, 'crowd_nav', 'configs', 'policy.config'))
    torch.manual_seed(0)
    env, robot, _ = make_env(human_num=5, test_sim='circle_crossing', policy_name='sarl', policy_config=pcfg)
    policy = robot.policy
    rows = []

    def maps_for(states, tag, extra=None):
        for cell_num, cell_size in ((4, 1.0), (6, 0.5), (8, 0.75)):
            for ch in (1, 2, 3):
                policy.cell_num, policy.cell_size, policy.om_channel_size = cell_num, cell_size, ch
                om = policy.build_occupancy_maps(states)
                row = {'tag': tag, 'cell_num': cell_num, 'cell_size': cell_size, 'channels': ch,
                       'humans': [[R(h.px), R(h.py), R(h.vx), R(h.vy)] for h in states],
                       'maps': [[R(v) for v in r] for r in om.reshape(len(states), -1).tolist()]}
                if extra:
                    row.update(extra)
                rows.append(row)

    for case in (0, 3):
        ob = env.reset('test', case)
        orca_robot = ORCA()
        orca_robot.time_step = env.time_step
        for step in range(13):
            state = JointState(robot.get_full_state(), ob)
            action = orca_robot.predict(state)
            if step in (4, 12):
                maps_for(ob, 'scene case %d step %d' % (case, step))
                nxt, _, _, _ = env.onestep_lookahead(ActionXY(action.vx, action.vy))
                maps_for(nxt, 'lookahead case %d step %d' % (case, step), {'scene': scene(env), 'global_time': R(env.global_time)})
            ob, reward, done, info = env.step(ActionXY(action.vx, action.vy))
            if done:
                break
    rng = np.random.RandomState(7)
    for n in (3, 8, 20):
        for rep in range(3):
            states = [ObservableState(*rng.uniform(-2.5, 2.5, 2), *rng.uniform(-1, 1, 2), 0.3) for _ in range(n)]
            if rep == 2:        # a standing human (atan2(0, 0) = 0) among them
                states[0] = ObservableState(states[0].px, states[0].py, 0.0, 0.0, 0.3)
            maps_for(states, 'random N=%d #%d' % (n, rep))
    # OM-SARL decisions of the reference itself (policy.config [sarl] with_om = true, seed-0 weights): per-action values
    # reward + gamma^(dt v_pref) * V(rotate(next state) ++ occupancy maps of the next human states) and the greedy action
    pcfg.set('sarl', 'with_om', 'true')
    torch.manual_seed(0)
    env, robot, _ = make_env(human_num=5, test_sim='circle_crossing', policy_name='sarl', policy_config=pcfg)
    policy = robot.policy
    decisions = []
    for case in (0, 3, 7):
        ob = env.reset('test', case)
        orca_robot = ORCA()
        orca_robot.time_step = env.time_step
        for step in range(12):
            state = JointState(robot.get_full_state(), ob)
            if step % 4 == 0:
                np_state = np.random.get_state()
                chosen = policy.predict(state)
                np.random.set_state(np_state)
                decisions.append({'case': case, 'step': step, 'scene': scene(env), 'global_time': R(env.global_time),
                                  'action': [R(chosen.vx), R(chosen.vy)], 'values': [R(v) for v in policy.action_values]})
            action = orca_robot.predict(state)
            ob, reward, done, info = env.step(ActionXY(action.vx, action.vy))
            if done:
                break
    with gzip.open(os.path.join(OUT, 'occupancy_maps.json.gz'), 'wt') as f:
        json.dump({'rows': rows, 'om_sarl': {'seed': 0, 'gamma': policy.gamma, 'cell_num': policy.cell_num, 'cell_size': policy.cell_size,
                                            'om_channel_size': policy.om_channel_size, 'decisions': decisions}}, f, separators=(',', ':'))
    print('occupancy map rows', len(rows))


def run_policy_decisions():
    """Greedy decisions of the reference's own CADRL and LSTM-RL policies (seed-0 weights, policy.config defaults, query_env):
    per-action values reward + gamma^(dt v_pref) * V and the chosen action on scenes a few steps into test episodes."""
    out = {}
    for key, name, tweak in (('cadrl', 'cadrl', None), ('lstm_rl', 'lstm_rl', None),
                             ('lstm_rl_interaction', 'lstm_rl', ('lstm_rl', 'with_interaction_module', 'true'))):
        pcfg = configparser.RawConfigParser()
        pcfg.read(os.path.join(REF, 'crowd_nav', 'configs', 'policy.config'))
        if tweak:
            pcfg.set(*tweak)
        torch.manual_seed(0)
        env, robot, _ = make_env(human_num=5, test_sim='circle_crossing', policy_name=name, policy_config=pcfg)
        policy = robot.policy
        decisions = []
        for case in (0, 3, 7):
            ob = env.reset('test', case)
            orca_robot = ORCA()
            orca_robot.time_step = env.time_step
            for step in range(12):
                state = JointState(robot.get_full_state(), ob)
                if step % 4 == 0:
                    np_state = np.random.get_state()
                    chosen = policy.predict(JointState(robot.get_full_state(), list(ob)))
                    np.random.set_state(np_state)
                    decisions.append({'case': case, 'step': step, 'scene': scene(env), 'global_time': R(env.global_time),
                                      'action': [R(chosen.vx), R(chosen.vy)], 'values': [R(v) for v in policy.action_values]})
                action = orca_robot.predict(state)
                ob, reward, done, info = env.step(ActionXY(action.vx, action.vy))
                if done:
                    break
        out[key] = {'seed': 0, 'gamma': policy.gamma, 'decisions': decisions}
        print(key, 'decisions', len(decisions))
    with gzip.open(os.path.join(OUT, 'policy_decisions.json.gz'), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))


def run_rl_memory():
    """Explorer.update_memory in RL mode (explorer.py:107-113), the reference's own method: value = reward +
    gamma^(dt v_pref) * target_model(next state), the reward alone on the terminal step, for every step of the episodes that
    end in success or collision (explorer.py:66-69). The episodes are the ORCA robot's test cases 0..7; the stored states are
    MultiHumanRL.transform(JointState) of a SARL policy (seed-0 weights, policy.config defaults) whose network is also the
    target model. (A randomly initialised SARL robot never ends an episode other than by timeout -- 40 of 40 train cases --
    and timeouts are not stored, so the robot that moves is ORCA; update_memory itself is called exactly as run_k_episodes
    calls it.)"""
    pcfg = configparser.RawConfigParser()
    pcfg.read(os.path.join(REF, 'crowd_nav', 'configs', 'policy.config'))
    torch.manual_seed(0)
    sarl = policy_factory['sarl'](); sarl.configure(pcfg); sarl.set_device(torch.device('cpu')); sarl.set_phase('test')
    env, robot, _ = make_env(human_num=5, test_sim='circle_crossing')

    class ListMemory(list):
        def push(self, item):
            self.append(item)
    mem = ListMemory()
    gamma = sarl.gamma
    explorer = Explorer(env, robot, torch.device('cpu'), memory=mem, gamma=gamma, target_policy=sarl)
    explorer.update_target_model(sarl.get_model())
    episodes = []
    for case in range(8):
        ob = env.reset('test', case)
        states, rewards, done = [], [], False
        while not done:
            states.append(sarl.transform(JointState(robot.get_full_state(), ob)))
            ob, reward, done, info = env.step(robot.act(ob))
            rewards.append(reward)
        n0 = len(mem)
        if isinstance(info, (ReachGoal, Collision)):
            explorer.update_memory(states, None, rewards, imitation_learning=False)
        episodes.append({'case': case, 'info': INFO_CODE[type(info)], 'steps': len(rewards), 'stored': len(mem) - n0})
    out = {'seed': 0, 'gamma': gamma, 'episodes': episodes, 'pairs': len(mem),
           'values': [R(v.item()) for _, v in mem],
           'states': [[[R(x) for x in row] for row in st.tolist()] for st, _ in mem]}
    print('rl_memory pairs', len(mem), [(e['case'], e['info'], e['stored']) for e in episodes])
    with gzip.open(os.path.join(OUT, 'rl_update_memory.json.gz'), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))


def run_human_times():
    """CrowdSim.get_human_times (crowd_sim.py:209-249) of the reference itself, after ORCA-robot episodes that ended at the
    goal: the state the call starts from, the arrivals already recorded during the episode, and what the call returns /
    leaves behind (human_times, global_time, agent positions)."""
    rows = []
    for tag, kw, cases in (('circle5', dict(human_num=5, test_sim='circle_crossing'), range(0, 40)),
                           ('circle10_visible', dict(human_num=10, test_sim='circle_crossing', robot_visible=True), range(0, 6)),
                           ('square20', dict(human_num=20, test_sim='square_crossing'), range(0, 30))):
        env, robot, _ = make_env(**kw)
        got = 0
        for case in cases:
            ob = env.reset('test', case)
            done = False
            while not done:
                ob, reward, done, info = env.step(robot.act(ob))
            if not isinstance(info, ReachGoal) or not robot.reached_destination():
                continue
            pre = scene(env)
            before = [R(t) for t in env.human_times]
            t0 = env.global_time
            times = env.get_human_times()
            rows.append({'tag': tag, 'case': case, 'N': kw['human_num'], 'robot_visible': bool(kw.get('robot_visible', False)),
                         'scene': pre, 'global_time': R(t0), 'human_times_before': before,
                         'human_times': [R(t) for t in times], 'global_time_after': R(env.global_time),
                         'final_robot': [R(robot.px), R(robot.py)], 'final_humans': [[R(h.px), R(h.py)] for h in env.humans]})
            got += 1
            if got >= (6 if tag == 'circle5' else 3):
                break
        print('human_times', tag, got)
    with gzip.open(os.path.join(OUT, 'human_times.json.gz'), 'wt') as f:
        json.dump({'rows': rows}, f, separators=(',', ':'))


NETWORK_PORTS = (  # name, the reference's module with the policy.config defaults (crowd_nav/policy/*.py)
    ('lstm_rl_v1', lambda: lstm_rl.ValueNetwork1(13, 6, [150, 100, 100, 1], 50)),
    ('lstm_rl_v2', lambda: lstm_rl.ValueNetwork2(13, 6, [150, 100, 100, 50], [150, 100, 100, 1], 50)),
    ('sarl', lambda: sarl.ValueNetwork(13, 6, [150, 100], [100, 50], [150, 100, 100, 1], [100, 100, 1], True, 1.0, 4)),
    ('cadrl', lambda: cadrl.ValueNetwork(13, [150, 100, 100, 1])),
)


def run_network_ports():
    """Outputs of the reference's value-network modules (LSTM-RL without / with interaction module, SARL, CADRL) with
    seeded stand-in weights loaded (network_port_weights), on a seeded input; CADRL sees the first human's rows only."""
    x = network_port_input()
    out = {}
    for i, (name, make) in enumerate(NETWORK_PORTS):
        net = make()
        keys_shapes = [(k, list(v.shape)) for k, v in net.state_dict().items()]
        net.load_state_dict(network_port_weights(keys_shapes, 100 + i))
        with torch.no_grad():
            y = net(x[:, 0] if name == 'cadrl' else x)
        out[name] = {'seed': 100 + i, 'keys_shapes': keys_shapes, 'output': [[R(v) for v in row] for row in y.tolist()]}
    with gzip.open(os.path.join(OUT, 'network_ports.json.gz'), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))
    print('network ports', {k: len(v['keys_shapes']) for k, v in out.items()})


def main():
    if '--network-ports-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_network_ports()
        return
    if '--human-times-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_human_times()
        return
    if '--rl-memory-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_rl_memory()
        return
    if '--policies-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_policy_decisions()
        return
    if '--mixed-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_mixed()
        run_resets()
        return
    if '--om-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_om()
        return
    if '--rotate-only' in sys.argv:
        os.makedirs(OUT, exist_ok=True)
        run_rotate()
        return
    quick = '--quick' in sys.argv
    os.makedirs(OUT, exist_ok=True)
    n = 50 if quick else 500
    run_suite('circle5_invisible', list(range(n)), human_num=5, test_sim='circle_crossing', record_traj=(0, 3, 118))
    run_suite('square5_invisible', list(range(n)), human_num=5, test_sim='square_crossing', record_traj=(0, 192))
    run_suite('square20_invisible', list(range(20 if quick else 100)), human_num=20, test_sim='square_crossing',
              record_traj=(0, 61))
    run_suite('circle5_visible', list(range(n)), human_num=5, test_sim='circle_crossing', robot_visible=True,
              record_traj=(1,))
    run_suite('circle10_visible', list(range(20 if quick else 100)), human_num=10, test_sim='circle_crossing',
              robot_visible=True)
    run_suite('circle5_random_attr', list(range(20 if quick else 100)), human_num=5, test_sim='circle_crossing',
              randomize=True, fresh_robot_sim=True)
    run_mixed()
    run_resets()
    run_rotate()
    run_om()
    run_policy_decisions()
    run_rl_memory()
    run_human_times()
    run_network_ports()


if __name__ == '__main__':
    main()
