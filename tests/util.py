import gzip
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def load_golden(name):
    with gzip.open(os.path.join(GOLDEN, name + '.json.gz'), 'rt') as f:
        return json.load(f)


SUITES = {
    # name: (N, rule, robot_visible, randomize_attributes)
    'circle5_invisible': (5, 'circle_crossing', 0, False),
    'square5_invisible': (5, 'square_crossing', 0, False),
    'square20_invisible': (20, 'square_crossing', 0, False),
    'circle5_visible': (5, 'circle_crossing', 1, False),
    'circle10_visible': (10, 'circle_crossing', 1, False),
    'circle5_random_attr': (5, 'circle_crossing', 0, True),
    'mixed5_invisible': (5, 'mixed', 0, False),      # 1..5 humans per case; unused slots are parked (crowdsim_b200.h)
}

PARKED_X = 1.0e6


def scene_arrays(scene, N=None):
    """robot [9], humans [n][8] (px,py,vx,vy,gx,gy,radius,v_pref). With N: padded to N rows with PARKED humans, the
    fixed-N layout's stand-in for humans a `mixed` scene does not have."""
    r = np.array([float(x) for x in scene['robot']])
    rows = [[float(x) for x in row] for row in scene['humans']]
    if N is not None:
        for i in range(len(rows), N):
            x = PARKED_X + 100.0 * i
            rows.append([x, PARKED_X, 0.0, 0.0, x, PARKED_X, 0.3, 1.0])
    h = np.array(rows)
    return r, h


def fill_host_state(po, scenes, N):
    """HostState with env e <- scenes[e] (golden 'scene' dicts)."""
    st = po.HostState(len(scenes), N)
    for e, sc in enumerate(scenes):
        st.set_scene(e, sc)
    return st


def network_port_weights(keys_shapes, seed):
    """Seeded weights for a state_dict layout [(key, shape)]: float32 uniform(-0.2, 0.2), one numpy RandomState draw per
    key in the given order (golden network_ports: loaded into the reference's modules and into the ports alike)."""
    import torch
    rng = np.random.RandomState(seed)
    return {k: torch.from_numpy(rng.uniform(-0.2, 0.2, shape).astype(np.float32)) for k, shape in keys_shapes}


def network_port_input():
    """[9 states][5 humans][13] float32 rows for the value networks (golden network_ports)."""
    import torch
    return torch.from_numpy(np.random.RandomState(12345).standard_normal((9, 5, 13)).astype(np.float32))


def ulp_diff(a, b):
    """Elementwise distance in float64 ulps (for values of equal sign / finite)."""
    a = np.ascontiguousarray(a, dtype=np.float64); b = np.ascontiguousarray(b, dtype=np.float64)
    ia = a.view(np.int64); ib = b.view(np.int64)
    return np.abs(ia - ib)
