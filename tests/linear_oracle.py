"""numpy front-end of tests/native/linear_oracle.c: the CPU oracle with crowdsim_params.human_policy and CROWDSIM_ROBOT_LINEAR
(TEST INFRASTRUCTURE). Same host arrays and structs as oracle/pyoracle.py (HostState, HostStepIO, HostEpisodes, reset); the
library is compiled with gcc into a temporary directory on first use."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import pyoracle as po
from crowdnav_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCE = os.path.join(ROOT, 'tests', 'native', 'linear_oracle.c')
CFLAGS = ['-O2', '-ffp-contract=off', '-fno-fast-math', '-fPIC', '-shared', '-std=gnu99', '-Wall', '-Wno-unused-function', '-fopenmp']

_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(tempfile.mkdtemp(prefix='linear_oracle_'), 'liblinear_oracle.so')
        subprocess.check_call(['gcc'] + CFLAGS + [SOURCE, '-o', so, '-lm'])
        l = C.CDLL(so)
        P = C.POINTER
        l.linear_oracle_step.restype = C.c_int
        l.linear_oracle_step.argtypes = [P(_abi.Params), C.c_int, C.c_int, P(_abi.State), P(_abi.StepIO), P(_abi.Episodes),
                                         P(_abi.AutoReset)]
        l.linear_oracle_lookahead_pack.restype = C.c_int
        l.linear_oracle_lookahead_pack.argtypes = [P(_abi.Params), C.c_int, C.c_int, P(_abi.State), C.c_void_p, C.c_int, C.c_int,
                                                   C.c_void_p, C.c_void_p]
        _lib = l
    return _lib


def step_rc(prm, st, io, ep=None, ar=None):
    s, i = st.struct(), io.struct()
    e = ep.struct() if ep is not None else None
    a = ar.struct() if ar is not None else None
    return lib().linear_oracle_step(C.byref(prm), st.B, st.N, C.byref(s), C.byref(i), C.byref(e) if e is not None else None,
                                    C.byref(a) if a is not None else None)


def step(prm, st, io, ep=None, ar=None):
    rc = step_rc(prm, st, io, ep, ar)
    assert rc == 0, rc


def run_episodes(prm, N, seeds, rule='circle_crossing', gamma=0.9, robot_v_pref=1.0, max_steps=200, **reset_kw):
    """One episode per seed to termination (lockstep, finished envs frozen): HostEpisodes + final state."""
    B = len(seeds)
    st = po.HostState(B, N); io = po.HostStepIO(B); ep = po.HostEpisodes(B, B, gamma, prm.time_step, robot_v_pref)
    ep.ep_case[:] = np.arange(B)
    po.reset(st, seeds, rule, ep=ep, robot_v_pref=robot_v_pref, **reset_kw)
    for _ in range(max_steps):
        if not st.active.any():
            break
        step(prm, st, io, ep)
    assert not st.active.any()
    return ep, st


def lookahead_pack(prm, st, actions, unicycle=False):
    actions = np.ascontiguousarray(actions, dtype=np.float64); A = actions.shape[0]
    states = np.zeros((st.B, A, st.N, 13), dtype=np.float32); reward = np.zeros((st.B, A)); s = st.struct()
    rc = lib().linear_oracle_lookahead_pack(C.byref(prm), st.B, st.N, C.byref(s), actions.ctypes.data, A, int(unicycle),
                                            states.ctypes.data, reward.ctypes.data)
    assert rc == 0, rc
    return states, reward


def lookahead_humans(prm, st):
    """The observation of env.onestep_lookahead: one step on a COPY of the state (it does not depend on the robot's action)."""
    cp = st.copy()
    step(prm, cp, po.HostStepIO(st.B))
    return cp.h_pos.copy(), cp.h_vel.copy()
