"""ctypes view of include/crowdsim_b200.h (the C ABI of libcrowdsim_b200.so).

The structs here are plain pointer/size carriers: the product fills them with DEVICE pointers
(`tensor.data_ptr()`); the test oracle (oracle/pyoracle.py) fills the same structs with host pointers
for its CPU library. No torch types cross the boundary.
"""
import ctypes as C
import os

ABI_VERSION = 5
MAX_HUMANS = 63
MAX_NEIGHBORS = 10

INFO_NOTHING, INFO_DANGER, INFO_REACHGOAL, INFO_COLLISION, INFO_TIMEOUT = 0, 1, 2, 3, 4
ROBOT_EXTERNAL_XY, ROBOT_ORCA, ROBOT_EXTERNAL_ROT, ROBOT_LINEAR = 0, 1, 2, 3
HUMANS_ORCA, HUMANS_LINEAR = 0, 1   # crowdsim_params.human_policy (env.config [humans] policy)
HUMAN_POLICIES = {'orca': HUMANS_ORCA, 'linear': HUMANS_LINEAR}
RULE_CIRCLE, RULE_SQUARE = 0, 1
RULE_MIXED = 2
PARKED_X = 1.0e6                  # include/crowdsim_b200.h: CROWDSIM_PARKED_X
RULES = {'circle_crossing': RULE_CIRCLE, 'square_crossing': RULE_SQUARE, 'mixed': RULE_MIXED}

_dp, _u8p, _i32p, _u32p, _f32p = (C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int32),
                                  C.POINTER(C.c_uint32), C.POINTER(C.c_float))


class Params(C.Structure):
    _fields_ = [('time_step', C.c_double), ('time_limit', C.c_double), ('success_reward', C.c_double),
                ('collision_penalty', C.c_double), ('discomfort_dist', C.c_double),
                ('discomfort_penalty_factor', C.c_double), ('neighbor_dist', C.c_double),
                ('time_horizon', C.c_double), ('max_neighbors', C.c_int32),
                ('human_safety_space', C.c_double), ('robot_safety_space', C.c_double),
                ('robot_visible', C.c_int32), ('robot_policy', C.c_int32),
                ('human_policy', C.c_int32)]       # last: the 13-argument positional form keeps meaning ORCA humans


class State(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('h_pos', 'h_vel', 'h_goal', 'h_attr', 'r_pos', 'r_vel', 'r_goal',
                                          'r_attr', 'r_theta', 'g_time', 'active')]


class StepIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('action', 'action_out', 'reward', 'dmin', 'done', 'info', 'obs32')]


class Episodes(C.Structure):
    _fields_ = [('ep_case', C.c_void_p), ('ep_steps', C.c_void_p), ('ep_return', C.c_void_p),
                ('ep_too_close', C.c_void_p), ('ep_min_dist_sum', C.c_void_p), ('discount', C.c_void_p),
                ('discount_len', C.c_int32),
                ('res_info', C.c_void_p), ('res_steps', C.c_void_p), ('res_time', C.c_void_p),
                ('res_return', C.c_void_p), ('res_too_close', C.c_void_p), ('res_min_dist_sum', C.c_void_p),
                ('res_final_rpos', C.c_void_p)]


class ResetArgs(C.Structure):
    _fields_ = [('mask', C.c_void_p), ('seed', C.c_void_p), ('seed_stride', C.c_uint32), ('rule', C.c_int32),
                ('circle_radius', C.c_double), ('square_width', C.c_double), ('human_radius', C.c_double),
                ('human_v_pref', C.c_double), ('robot_radius', C.c_double), ('robot_v_pref', C.c_double),
                ('discomfort_dist', C.c_double), ('randomize_attributes', C.c_int32),
                ('case_counter', C.c_void_p), ('case_total', C.c_int32),
                ('seed_base', C.c_uint32), ('case_first', C.c_int32), ('case_wrap', C.c_int32)]


class AutoReset(C.Structure):
    _fields_ = [('n_h_pos', C.c_void_p), ('n_h_goal', C.c_void_p), ('n_h_attr', C.c_void_p), ('n_case', C.c_void_p),
                ('n_state', C.c_void_p), ('want', C.c_void_p), ('circle_radius', C.c_double),
                ('robot_radius', C.c_double), ('robot_v_pref', C.c_double)]


SLOT_EMPTY, SLOT_READY, SLOT_EXHAUSTED = 0, 1, 2


def declare(lib, prefix='crowdsim_', with_stream=True):
    """Attach argtypes/restype for the compute entry points (shared by product and oracle libs)."""
    s = [C.c_void_p] if with_stream else []
    P = C.POINTER
    f = getattr(lib, prefix + 'step')
    f.restype, f.argtypes = C.c_int, [P(Params), C.c_int, C.c_int, P(State), P(StepIO), P(Episodes), P(AutoReset)] + s
    if hasattr(lib, prefix + 'step_n'):
        f = getattr(lib, prefix + 'step_n')
        f.restype, f.argtypes = C.c_int, [P(Params), C.c_int, C.c_int, P(State), P(StepIO), P(Episodes), P(AutoReset), C.c_int] + s
    f = getattr(lib, prefix + 'prefetch_scenes')
    f.restype, f.argtypes = C.c_int, [P(ResetArgs), C.c_int, C.c_int, P(AutoReset)] + s
    f = getattr(lib, prefix + 'orca_act')
    f.restype, f.argtypes = C.c_int, [P(Params), C.c_int, C.c_int, P(State), C.c_void_p] + s
    f = getattr(lib, prefix + 'reset')
    f.restype, f.argtypes = C.c_int, [P(ResetArgs), C.c_int, C.c_int, P(State), P(Episodes)] + s
    f = getattr(lib, prefix + 'pack_joint')
    f.restype, f.argtypes = C.c_int, [C.c_int, C.c_int, P(State), C.c_int, C.c_void_p] + s
    f = getattr(lib, prefix + 'lookahead_pack')
    f.restype, f.argtypes = C.c_int, [P(Params), C.c_int, C.c_int, P(State), C.c_void_p, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p] + s
    return lib


EXPORTS = ('crowdsim_abi_version', 'crowdsim_device_check', 'crowdsim_launch_count', 'crowdsim_debug_force_generic', 'crowdsim_graph_launch',
           'crowdsim_event_wait', 'crowdsim_host_pump', 'crowdsim_step', 'crowdsim_step_n',
           'crowdsim_orca_act', 'crowdsim_reset', 'crowdsim_prefetch_scenes', 'crowdsim_pack_joint', 'crowdsim_lookahead_pack',
           'crowdsim_lookahead_humans', 'crowdsim_occupancy_maps', 'crowdsim_human_times', 'crowdsim_onestep_lookahead')

# CROWDSIM_B200_LIB selects another build of the SAME library (A/B runs of kernel variants, scripts/gpu_variants.sh);
# it is never a fallback: the named file must exist.
LIB_PATH = os.environ.get('CROWDSIM_B200_LIB') or os.path.join(os.path.dirname(os.path.abspath(__file__)), 'csrc',
                                                               'libcrowdsim_b200.so')
_lib = None


class CudaLibraryMissing(RuntimeError):
    pass


def load():
    """Load libcrowdsim_b200.so. There is NO CPU fallback: a missing library is an error."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CudaLibraryMissing(
                'libcrowdsim_b200.so is not built (%s). Run `python -m crowdnav_b200.build` '
                '(needs nvcc); the product path has no CPU fallback.' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.crowdsim_abi_version.restype = C.c_int
        lib.crowdsim_device_check.restype = C.c_int
        lib.crowdsim_device_check.argtypes = [C.POINTER(C.c_int)] * 3
        lib.crowdsim_launch_count.restype = C.c_ulonglong
        lib.crowdsim_debug_force_generic.argtypes = [C.c_int]
        lib.crowdsim_debug_force_generic.restype = None
        lib.crowdsim_graph_launch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crowdsim_graph_launch.restype = C.c_int
        lib.crowdsim_event_wait.argtypes = [C.c_void_p]
        lib.crowdsim_event_wait.restype = C.c_int
        lib.crowdsim_host_pump.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
        lib.crowdsim_host_pump.restype = C.c_int
        lib.crowdsim_lookahead_humans.argtypes = [C.POINTER(Params), C.c_int, C.c_int, C.POINTER(State), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crowdsim_lookahead_humans.restype = C.c_int
        lib.crowdsim_occupancy_maps.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
        lib.crowdsim_occupancy_maps.restype = C.c_int
        lib.crowdsim_human_times.argtypes = [C.POINTER(Params), C.c_int, C.c_int, C.POINTER(State), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        lib.crowdsim_human_times.restype = C.c_int
        lib.crowdsim_onestep_lookahead.argtypes = [C.POINTER(Params), C.c_int, C.c_int, C.POINTER(State), C.POINTER(StepIO), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crowdsim_onestep_lookahead.restype = C.c_int
        declare(lib)
        if lib.crowdsim_abi_version() != ABI_VERSION:
            raise CudaLibraryMissing('ABI version mismatch: library %d, python %d'
                                     % (lib.crowdsim_abi_version(), ABI_VERSION))
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        if rc > 0:
            raise RuntimeError('%s: CUDA error %d' % (what, rc))
        raise ValueError('%s: %s' % (what, {-1: 'invalid argument', -2: 'unsupported size or policy',
                                             -3: 'no sm_100 CUDA device'}.get(rc, 'error %d' % rc)))
