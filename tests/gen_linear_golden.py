#!/usr/bin/env python
"""Generate the Linear-policy fixtures (tests/golden/*linear*) by running the REFERENCE'S OWN PYTHON, unmodified.

TEST INFRASTRUCTURE, run in the build container like oracle/gen_golden.py, whose environment set-up, suite driver and
recording format it reuses (imported as a module; the reference with oracle/shims on sys.path).

  python tests/gen_linear_golden.py [--quick] [--out DIR]

The Linear policy (crowd_sim/envs/policy/linear.py) for the humans (env.config [humans] policy = linear) and / or the robot
(test.py --policy linear): test suites with the reference Explorer's log lines and trajectories, and the greedy decisions of
the reference's SARL / CADRL (seed-0 weights) among linear humans.

The reference's CrowdSim.configure raises NotImplementedError for any [humans] policy but orca (crowd_sim.py:60-70), although
the humans it creates at every reset take their policy from the same config object (agent.py:19, crowd_sim.py:101-151): the
driver selects Linear humans on that config after configure.
"""
import configparser
import gzip
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), 'oracle'))

import gen_golden as G  # noqa: E402  (builds the oracle libraries, imports the reference)

_make_env = G.make_env


def make_env(human_policy='orca', **kw):
    env, robot, cfg = _make_env(**kw)
    cfg.set('humans', 'policy', human_policy)      # read by every Human created from now on (agent.py:19)
    return env, robot, cfg


G.make_env = make_env          # run_suite builds its environments through the module's make_env


def run_decisions():
    """SARL / CADRL greedy decisions (per-action values and action) a few steps into test episodes among linear humans,
    the robot driven by ORCA in between (like gen_golden.run_policy_decisions)."""
    out = {}
    for key in ('cadrl', 'sarl'):
        pcfg = configparser.RawConfigParser()
        pcfg.read(os.path.join(G.REF, 'crowd_nav', 'configs', 'policy.config'))
        G.torch.manual_seed(0)
        env, robot, _ = make_env(human_num=5, test_sim='circle_crossing', policy_name=key, policy_config=pcfg, human_policy='linear')
        policy = robot.policy
        decisions = []
        for case in (0, 3, 7):
            ob = env.reset('test', case)
            orca_robot = G.ORCA()
            orca_robot.time_step = env.time_step
            for step in range(12):
                state = G.JointState(robot.get_full_state(), ob)
                if step % 4 == 0:
                    np_state = G.np.random.get_state()
                    chosen = policy.predict(G.JointState(robot.get_full_state(), list(ob)))
                    G.np.random.set_state(np_state)
                    decisions.append({'case': case, 'step': step, 'scene': G.scene(env), 'global_time': G.R(env.global_time),
                                      'action': [G.R(chosen.vx), G.R(chosen.vy)], 'values': [G.R(v) for v in policy.action_values]})
                action = orca_robot.predict(state)
                ob, reward, done, info = env.step(G.ActionXY(action.vx, action.vy))
                if done:
                    break
        out[key] = {'seed': 0, 'gamma': policy.gamma, 'decisions': decisions}
        print('linear humans', key, 'decisions', len(decisions))
    with gzip.open(os.path.join(G.OUT, 'policy_decisions_linear_humans.json.gz'), 'wt') as f:
        json.dump(out, f, separators=(',', ':'))


def main():
    if '--out' in sys.argv:
        G.OUT = sys.argv[sys.argv.index('--out') + 1]
    os.makedirs(G.OUT, exist_ok=True)
    n = 50 if '--quick' in sys.argv else 500
    G.run_suite('circle5_linear_humans_invisible', list(range(n)), human_num=5, test_sim='circle_crossing', human_policy='linear',
                record_traj=(0, 3))
    G.run_suite('circle5_linear_humans_visible', list(range(n)), human_num=5, test_sim='circle_crossing', human_policy='linear',
                robot_visible=True, record_traj=(1,))
    G.run_suite('circle5_linear_robot', list(range(n)), human_num=5, test_sim='circle_crossing', policy_name='linear',
                record_traj=(0, 2))
    G.run_suite('circle5_linear_both', list(range(n)), human_num=5, test_sim='circle_crossing', policy_name='linear',
                human_policy='linear', record_traj=(0,))
    G.run_suite('square20_linear_humans', list(range(20 if n == 50 else 100)), human_num=20, test_sim='square_crossing',
                human_policy='linear', record_traj=(0,))
    G.run_suite('mixed5_linear_humans', list(range(300)), human_num=5, test_sim='mixed', human_policy='linear', reset_human_num=5,
                record_traj=(1, 4, 8))
    run_decisions()


if __name__ == '__main__':
    main()
