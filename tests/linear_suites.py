"""The Linear-policy fixtures (tests/golden/*linear*, tests/gen_linear_golden.py) and the parameters they were made with."""

# name: (N, rule, robot_visible, robot policy, human policy)
LINEAR_SUITES = {
    'circle5_linear_humans_invisible': (5, 'circle_crossing', 0, 'orca', 'linear'),
    'circle5_linear_humans_visible': (5, 'circle_crossing', 1, 'orca', 'linear'),
    'circle5_linear_robot': (5, 'circle_crossing', 0, 'linear', 'orca'),
    'circle5_linear_both': (5, 'circle_crossing', 0, 'linear', 'linear'),
    'square20_linear_humans': (20, 'square_crossing', 0, 'orca', 'linear'),
    'mixed5_linear_humans': (5, 'mixed', 0, 'orca', 'linear'),    # unused human slots are parked (crowdsim_b200.h)
}

TOL = 1e-12     # float64 state / reward / return bar against the reference (numpy's scalar arctan2 is not glibc's atan2)


def params(oracle, name, **over):
    """crowdsim_params of a fixture suite (oracle.default_params + the suite's visibility and policies)."""
    from crowdnav_b200 import _abi
    _, _, vis, robot, humans = LINEAR_SUITES[name]
    kw = dict(robot_visible=vis, robot_policy=_abi.ROBOT_LINEAR if robot == 'linear' else _abi.ROBOT_ORCA,
              human_policy=_abi.HUMAN_POLICIES[humans])
    kw.update(over)
    return oracle.default_params(**kw)
