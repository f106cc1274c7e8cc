"""The fixtures of non-default configurations (tests/gen_config_golden.py) and the parameters that reproduce them, for the CPU
oracle (oracle/pyoracle.py) and for BatchedCrowdSim."""
# env.config values of the `shift` configuration: a time step that is not a power of two, every reward / scene / agent
# constant moved off its default
SHIFT_PARAMS = dict(time_step=0.1, time_limit=30.0, success_reward=2.0, collision_penalty=-0.5, discomfort_dist=0.25,
                    discomfort_penalty_factor=0.8)
SHIFT_RESET = dict(circle_radius=5.0, square_width=12.0, human_radius=0.25, human_v_pref=1.2, robot_radius=0.35,
                   robot_v_pref=0.8, discomfort_dist=0.25)
SHIFT_CONFIG = (('env', 'time_step', '0.1'), ('env', 'time_limit', '30'),
                ('reward', 'success_reward', '2'), ('reward', 'collision_penalty', '-0.5'), ('reward', 'discomfort_dist', '0.25'),
                ('reward', 'discomfort_penalty_factor', '0.8'), ('sim', 'circle_radius', '5'), ('sim', 'square_width', '12'),
                ('humans', 'radius', '0.25'), ('humans', 'v_pref', '1.2'), ('robot', 'radius', '0.35'), ('robot', 'v_pref', '0.8'))
CONFIGS = {'default': ({}, {}, ()), 'shift': (SHIFT_PARAMS, SHIFT_RESET, SHIFT_CONFIG)}

CONFIG_SUITES = {
    # name: (N, rule, robot_visible, phase, configuration, robot ORCA safety_space)
    'il5_train': (5, 'circle_crossing', 0, 'train', 'default', 0.15),      # train.py's imitation-learning demonstrations
    'shift5_circle': (5, 'circle_crossing', 0, 'test', 'shift', 0.0),
    'shift5_square': (5, 'square_crossing', 0, 'test', 'shift', 0.0),
    'shift10_visible': (10, 'circle_crossing', 1, 'test', 'shift', 0.0),
}
TRAJ_SUITES = ('il5_train', 'shift5_circle', 'shift5_square')
PHASE_OFFSET = {'train': 2000, 'val': 0, 'test': 1000}


def params(oracle, name, **over):
    N, rule, vis, phase, config, safety = CONFIG_SUITES[name]
    p = dict(CONFIGS[config][0], robot_visible=vis, robot_safety_space=safety)
    p.update(over)
    return oracle.default_params(**p)


def reset_kw(name):
    return dict(CONFIGS[CONFIG_SUITES[name][4]][1])


def seeds(name, cases):
    return [PHASE_OFFSET[CONFIG_SUITES[name][3]] + c['case'] for c in cases]


def time_limit(name):
    return CONFIGS[CONFIG_SUITES[name][4]][0].get('time_limit', 25.0)


def time_step(name):
    return CONFIGS[CONFIG_SUITES[name][4]][0].get('time_step', 0.25)


def max_steps(name):
    from crowdnav_b200.batched import max_episode_steps
    return max_episode_steps(time_limit(name), time_step(name))


def env_config(config='default', **kw):
    """BatchedCrowdSim config: batched.default_config(**kw) with the configuration's overrides."""
    from crowdnav_b200.batched import default_config
    cfg = default_config(**kw)
    for section, key, value in CONFIGS[config][2]:
        cfg.set(section, key, value)
    return cfg


def pre_times(steps):
    """global_time before each recorded step of a trajectory (that of the previous step's end; 0 at the start)."""
    return [0.0] + [float(s['global_time']) for s in steps[:-1]]
