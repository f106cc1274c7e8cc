#!/usr/bin/env python
"""Generate the fixtures of non-default configurations (tests/golden/*il5_train*, *shift*) by running the REFERENCE'S OWN
PYTHON, unmodified.

TEST INFRASTRUCTURE, run in the build container like oracle/gen_golden.py, whose environment set-up, suite driver and
recording format it reuses (imported as a module; the reference with oracle/shims on sys.path).

  python tests/gen_config_golden.py [--out DIR]

Two configurations besides the defaults every other fixture uses:
  il5_train  train.py's imitation-learning demonstrations (train.py:117-129, train.config [imitation_learning]): train phase,
             an ORCA robot with safety_space = 0.15 and multiagent_training = True, invisible robot, env.config defaults.
  shift      a time step that is not a power of two and every reward, scene and agent constant moved off its default
             (SHIFT below), test phase.
The wrapped make_env applies the overrides to the config, configures the env again and creates the Robot from the
overridden config; it sets the ORCA robot's safety_space / multiagent_training after gen_golden.make_env, which zeroes
safety_space.
"""
import gzip
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), 'oracle'))

import gen_golden as G  # noqa: E402  (builds the oracle libraries, imports the reference)

_make_env = G.make_env

SHIFT = (('env', 'time_step', '0.1'), ('env', 'time_limit', '30'),
         ('reward', 'success_reward', '2'), ('reward', 'collision_penalty', '-0.5'), ('reward', 'discomfort_dist', '0.25'),
         ('reward', 'discomfort_penalty_factor', '0.8'), ('sim', 'circle_radius', '5'), ('sim', 'square_width', '12'),
         ('humans', 'radius', '0.25'), ('humans', 'v_pref', '1.2'), ('robot', 'radius', '0.35'), ('robot', 'v_pref', '0.8'))
CONFIGS = {'default': (), 'shift': SHIFT}


def make_env(config='default', safety_space=0.0, multiagent_training=None, **kw):
    env, robot, cfg = _make_env(**kw)
    test_sim = env.test_sim
    for section, key, value in CONFIGS[config]:
        cfg.set(section, key, value)
    env.configure(cfg)
    env.test_sim = test_sim
    policy = robot.policy
    robot = G.Robot(cfg, 'robot')
    robot.set_policy(policy)
    env.set_robot(robot)
    if isinstance(policy, G.ORCA):
        policy.safety_space = safety_space
        policy.multiagent_training = multiagent_training
    return env, robot, cfg


G.make_env = make_env          # run_suite builds its environments through the module's make_env

IL = dict(config='default', safety_space=0.15, multiagent_training=True)


def run_human_times():
    """CrowdSim.get_human_times at the shift configuration, after ORCA-robot episodes that ended at the goal (like
    gen_golden.run_human_times)."""
    rows = []
    for tag, kw, cases in (('shift5', dict(human_num=5, test_sim='circle_crossing'), range(0, 40)),
                           ('shift10_visible', dict(human_num=10, test_sim='circle_crossing', robot_visible=True), range(0, 20))):
        env, robot, _ = make_env(config='shift', **kw)
        got = 0
        for case in cases:
            ob = env.reset('test', case)
            done = False
            while not done:
                ob, reward, done, info = env.step(robot.act(ob))
            if not isinstance(info, G.ReachGoal) or not robot.reached_destination():
                continue
            pre = G.scene(env)
            before = [G.R(t) for t in env.human_times]
            t0 = env.global_time
            times = env.get_human_times()
            rows.append({'tag': tag, 'case': case, 'N': kw['human_num'], 'robot_visible': bool(kw.get('robot_visible', False)),
                         'scene': pre, 'global_time': G.R(t0), 'human_times_before': before,
                         'human_times': [G.R(t) for t in times], 'global_time_after': G.R(env.global_time),
                         'final_robot': [G.R(robot.px), G.R(robot.py)], 'final_humans': [[G.R(h.px), G.R(h.py)] for h in env.humans]})
            got += 1
            if got >= 4:
                break
        print('human_times', tag, got)
    with gzip.open(os.path.join(G.OUT, 'human_times_shift.json.gz'), 'wt') as f:
        json.dump({'rows': rows}, f, separators=(',', ':'))


def run_il_memory(k=6):
    """The reference's Explorer.run_k_episodes(k, 'train', update_memory=True, imitation_learning=True) with the ORCA robot of
    train.py's demonstrations at the shift configuration: the (state, value) pairs update_memory pushes, states transformed by
    a SARL policy (seed-0 weights, policy.config defaults) as train.py's target policy does."""
    import configparser
    pcfg = configparser.RawConfigParser()
    pcfg.read(os.path.join(G.REF, 'crowd_nav', 'configs', 'policy.config'))
    G.torch.manual_seed(0)
    sarl = G.policy_factory['sarl'](); sarl.configure(pcfg); sarl.set_device(G.torch.device('cpu')); sarl.set_phase('train')
    env, robot, _ = make_env(config='shift', safety_space=0.15, multiagent_training=True, human_num=5, test_sim='circle_crossing')

    class ListMemory(list):
        def push(self, item):
            self.append(item)
    mem = ListMemory()
    explorer = G.Explorer(env, robot, G.torch.device('cpu'), memory=mem, gamma=sarl.gamma, target_policy=sarl)
    env.case_counter['train'] = 0
    explorer.run_k_episodes(k, 'train', update_memory=True, imitation_learning=True)
    out = {'seed': 0, 'gamma': sarl.gamma, 'k': k, 'pairs': len(mem),
           'values': [G.R(v.item()) for _, v in mem],
           'states': [[[G.R(x) for x in row] for row in st.tolist()] for st, _ in mem]}
    print('il_memory pairs', len(mem))
    with gzip.open(os.path.join(G.OUT, 'il_update_memory_shift.json.gz'), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))


def main():
    if '--out' in sys.argv:
        G.OUT = sys.argv[sys.argv.index('--out') + 1]
    os.makedirs(G.OUT, exist_ok=True)
    G.run_suite('il5_train', list(range(300)), phase='train', human_num=5, test_sim='circle_crossing', record_traj=(0, 7), **IL)
    G.run_suite('shift5_circle', list(range(300)), config='shift', human_num=5, test_sim='circle_crossing', record_traj=(0,))
    G.run_suite('shift5_square', list(range(300)), config='shift', human_num=5, test_sim='square_crossing', record_traj=(0,))
    G.run_suite('shift10_visible', list(range(100)), config='shift', human_num=10, test_sim='circle_crossing', robot_visible=True)
    run_human_times()
    run_il_memory()


if __name__ == '__main__':
    main()
