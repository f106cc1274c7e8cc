"""BatchedCrowdSim: B independent CrowdSim-v0 environments stepped in lockstep on one B200.

Host-side driver of libcrowdsim_b200.so (include/crowdsim_b200.h). torch is used only as plumbing: device
memory (float64 SoA tensors), streams, host<->device copies; every env-step is hand-written CUDA.

Mirrors the reference environment's surface for a batch (paths relative to /root/reference):
  configure(config)   crowd_sim/envs/crowd_sim.py:51-79   (same RawConfigParser sections/keys)
  reset(phase, ...)   crowd_sim/envs/crowd_sim.py:251-312 (per-case MT19937 seeding: offset[phase] + case)
  step(actions)       crowd_sim/envs/crowd_sim.py:317-420 -> (ob, reward, done, info) as tensors
  onestep_lookahead   crowd_sim/envs/crowd_sim.py:314-315 (batched over the 81-action space, fused with rotate)
There is no CPU fallback: without the CUDA library / a GPU these calls raise.
"""
import ctypes as C

import numpy as np
import torch

from . import _abi

_PHASE_OFFSET = {'train': 2000, 'val': 0, 'test': 1000}   # crowd_sim.py:270-271 (case_capacity val=test=1000)


def _ptr(t):
    return None if t is None else t.data_ptr()


def max_episode_steps(time_limit, time_step):
    """Steps an episode can last: the timeout fires on the first step with global_time >= time_limit - 1
    (crowd_sim.py:368; 97 with the default 25 s / 0.25 s). +2 of slack."""
    import math
    return int(math.ceil(float(time_limit) / float(time_step))) + 2


def discount_table(gamma, time_step, v_pref, n=128):
    """explorer.py:71-72: pow(gamma, t * time_step * v_pref) for t = 0..n-1, computed with C pow on the host so the
    device-side discounted return is bit-identical to the reference's. n must cover the longest episode
    (max_episode_steps): the kernels treat steps beyond the table as undiscounted-to-zero."""
    return [pow(gamma, t * time_step * v_pref) for t in range(n)]


class Slab(object):
    """One contiguous byte buffer carved into typed tensors (256-byte aligned). The arrays a host-side caller reads after
    every step (observation, reward, done, info, applied / next action) live in one slab so that ONE device->host copy
    moves them all (five separate copies cost ~2.5 us of per-copy overhead each on the e2e path)."""

    def __init__(self, layout, device, pin=False):
        """layout: list of (name, shape, dtype)."""
        self.layout, self.offsets, off = layout, {}, 0
        for name, shape, dtype in layout:
            n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
            self.offsets[name] = (off, n)
            off += (n + 255) // 256 * 256
        self.nbytes = off
        self.buf = torch.zeros(off, dtype=torch.uint8, device=device)
        if pin:
            self.buf = self.buf.pin_memory()
        self.views = {name: self.buf[self.offsets[name][0]:self.offsets[name][0] + self.offsets[name][1]].view(dtype).view(*shape)
                      for name, shape, dtype in layout}

    def __getitem__(self, name):
        return self.views[name]


def host_visible_layout(B, N):
    """Everything a host-side caller may read after a step, ordered so that both views are ONE contiguous range:
    compact view  = [obs32 .. next_action]   float32 observation (crowdsim_step_io.obs32) + reward, dmin, done, info
                    (+ the robot's next ORCA decision, produced by a later kernel): 114 B per env at N = 5
    float64 view  = [reward .. h_vel]        the same scalars + the float64 state arrays themselves: 210 B per env"""
    return [('obs32', (B, N, 4), torch.float32), ('reward', (B,), torch.float64), ('dmin', (B,), torch.float64),
            ('done', (B,), torch.uint8), ('info', (B,), torch.uint8), ('next_action', (B, 2), torch.float64),
            ('action_out', (B, 2), torch.float64), ('h_pos', (B, N, 2), torch.float64), ('h_vel', (B, N, 2), torch.float64),
            # the rest of the mutable state, so that a single-env caller mirrors everything with ONE copy of the slab (compat)
            ('r_pos', (B, 2), torch.float64), ('r_vel', (B, 2), torch.float64), ('r_theta', (B,), torch.float64), ('g_time', (B,), torch.float64)]


class DeviceState(object):
    """crowdsim_state on device tensors ([B][N][2] / [B][2] / [B] float64)."""
    FIELDS = ('h_pos', 'h_vel', 'h_goal', 'h_attr', 'r_pos', 'r_vel', 'r_goal', 'r_attr', 'r_theta', 'g_time')

    def __init__(self, B, N, device, slab=None):
        self.B, self.N, self.device = B, N, device
        z = lambda *s: torch.zeros(s, dtype=torch.float64, device=device)  # noqa: E731
        if slab is not None:
            self.h_pos, self.h_vel = slab['h_pos'], slab['h_vel']
            self.r_pos, self.r_vel, self.r_theta, self.g_time = slab['r_pos'], slab['r_vel'], slab['r_theta'], slab['g_time']
        else:
            self.h_pos, self.h_vel = z(B, N, 2), z(B, N, 2)
            self.r_pos, self.r_vel, self.r_theta, self.g_time = z(B, 2), z(B, 2), z(B), z(B)
        self.h_goal, self.h_attr = z(B, N, 2), z(B, N, 2)
        self.r_goal, self.r_attr = z(B, 2), z(B, 2)
        self.active = torch.ones(B, dtype=torch.uint8, device=device)

    def struct(self, with_active=True):
        return _abi.State(*[_ptr(getattr(self, f)) for f in self.FIELDS], _ptr(self.active) if with_active else None)

    def load_host(self, host):
        """Copy from an object with the same numpy fields (e.g. oracle.pyoracle.HostState in tests)."""
        for f in self.FIELDS:
            getattr(self, f).copy_(torch.from_numpy(np.ascontiguousarray(getattr(host, f))))
        if getattr(host, 'active', None) is not None:
            self.active.copy_(torch.from_numpy(host.active))

    def to_host(self):
        out = {f: getattr(self, f).cpu().numpy() for f in self.FIELDS}
        out['active'] = self.active.cpu().numpy()
        return out


class EpisodeBuffers(object):
    """crowdsim_episodes: slot accumulators + per-case results of Explorer.run_k_episodes (explorer.py:35-72)."""

    def __init__(self, B, k, device, gamma, time_step, v_pref, max_steps=128):
        i32 = lambda n, v=0: torch.full((n,), v, dtype=torch.int32, device=device)  # noqa: E731
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=device)  # noqa: E731
        self.k = k
        self.ep_case, self.ep_steps, self.ep_too_close = i32(B, -1), i32(B), i32(B)
        self.ep_return, self.ep_min_dist_sum = f64(B), f64(B)
        self.discount = torch.tensor(discount_table(gamma, time_step, v_pref, max(128, max_steps)), dtype=torch.float64, device=device)
        self.res_info = torch.zeros(k, dtype=torch.uint8, device=device)
        self.res_steps, self.res_too_close = i32(k), i32(k)
        self.res_time, self.res_return, self.res_min_dist_sum = f64(k), f64(k), f64(k)
        self.res_final_rpos = f64(k, 2)

    def struct(self):
        return _abi.Episodes(_ptr(self.ep_case), _ptr(self.ep_steps), _ptr(self.ep_return), _ptr(self.ep_too_close),
                             _ptr(self.ep_min_dist_sum), _ptr(self.discount), self.discount.numel(),
                             _ptr(self.res_info), _ptr(self.res_steps), _ptr(self.res_time), _ptr(self.res_return),
                             _ptr(self.res_too_close), _ptr(self.res_min_dist_sum), _ptr(self.res_final_rpos))


class AutoResetBuffers(object):
    """crowdsim_autoreset: one prefetched "next scene" slot per env (see include/crowdsim_b200.h)."""

    def __init__(self, B, N, device, circle_radius, robot_radius, robot_v_pref):
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=device)  # noqa: E731
        self.n_h_pos, self.n_h_goal, self.n_h_attr = f64(B, N, 2), f64(B, N, 2), f64(B, N, 2)
        self.n_case = torch.full((B,), -1, dtype=torch.int32, device=device)
        self.n_state = torch.zeros(B, dtype=torch.uint8, device=device)
        self.want = torch.zeros(B, dtype=torch.uint8, device=device)
        self.circle_radius, self.robot_radius, self.robot_v_pref = circle_radius, robot_radius, robot_v_pref

    FIELDS = ('n_h_pos', 'n_h_goal', 'n_h_attr', 'n_case', 'n_state', 'want')

    def struct(self):
        return _abi.AutoReset(_ptr(self.n_h_pos), _ptr(self.n_h_goal), _ptr(self.n_h_attr), _ptr(self.n_case),
                              _ptr(self.n_state), _ptr(self.want), self.circle_radius, self.robot_radius, self.robot_v_pref)

    def load_host(self, host):
        for f in self.FIELDS:
            getattr(self, f).copy_(torch.from_numpy(np.ascontiguousarray(getattr(host, f))))

    def to_host(self):
        return {f: getattr(self, f).cpu().numpy() for f in self.FIELDS}


class BatchedCrowdSim(object):
    def __init__(self, num_envs, device='cuda:0'):
        self.lib = _abi.load()
        if not torch.cuda.is_available():
            raise RuntimeError('BatchedCrowdSim needs a CUDA device (no CPU fallback)')
        self.device = torch.device(device)
        self.B = int(num_envs)
        # crowd_sim.py:26-49 attributes
        self.time_limit = None; self.time_step = None
        self.success_reward = None; self.collision_penalty = None
        self.discomfort_dist = None; self.discomfort_penalty_factor = None
        self.config = None; self.case_capacity = None; self.case_size = None; self.case_counter = None
        self.randomize_attributes = None; self.train_val_sim = None; self.test_sim = None
        self.square_width = None; self.circle_radius = None; self.human_num = None
        # robot / humans (agent.py:16-20 config keys)
        self.robot_visible = False; self.robot_radius = 0.3; self.robot_v_pref = 1.0
        self.human_radius = 0.3; self.human_v_pref = 1.0
        self.robot_policy = _abi.ROBOT_ORCA
        self.human_policy = _abi.HUMANS_ORCA
        self.human_safety_space = 0.0; self.robot_safety_space = 0.0
        # ORCA constants (orca.py:61-64)
        self.neighbor_dist = 10.0; self.max_neighbors = 10; self.time_horizon = 5.0
        self.state = None; self.episodes = None; self.autoreset = None
        self._case_counter = None; self._case_total = 0; self._seed_base = 0; self._case_first = 0; self._case_wrap = 0
        self._ar_rule = None; self._ar_seed_stride = 0

    # ---- configuration -------------------------------------------------------------------------------------------
    def configure(self, config):
        """Same keys as crowd_sim.py:51-68 plus the [humans]/[robot] agent attributes of agent.py:16-20."""
        self.config = config
        self.time_limit = config.getint('env', 'time_limit')
        self.time_step = config.getfloat('env', 'time_step')
        self.randomize_attributes = config.getboolean('env', 'randomize_attributes')
        self.success_reward = config.getfloat('reward', 'success_reward')
        self.collision_penalty = config.getfloat('reward', 'collision_penalty')
        self.discomfort_dist = config.getfloat('reward', 'discomfort_dist')
        self.discomfort_penalty_factor = config.getfloat('reward', 'discomfort_penalty_factor')
        # env.config [humans] policy (policy_factory.py:9-12): 'orca' or 'linear' (straight to the goal, ignores everyone)
        human_policy = config.get('humans', 'policy')
        if human_policy not in _abi.HUMAN_POLICIES:
            raise NotImplementedError
        self.human_policy = _abi.HUMAN_POLICIES[human_policy]
        u32max = int(np.iinfo(np.uint32).max)
        self.case_capacity = {'train': u32max - 2000, 'val': 1000, 'test': 1000}
        self.case_size = {'train': u32max - 2000, 'val': config.getint('env', 'val_size'),
                          'test': config.getint('env', 'test_size')}
        self.train_val_sim = config.get('sim', 'train_val_sim')
        self.test_sim = config.get('sim', 'test_sim')
        self.square_width = config.getfloat('sim', 'square_width')
        self.circle_radius = config.getfloat('sim', 'circle_radius')
        self.human_num = config.getint('sim', 'human_num')
        self.case_counter = {'train': 0, 'test': 0, 'val': 0}
        self.human_radius = config.getfloat('humans', 'radius')
        self.human_v_pref = config.getfloat('humans', 'v_pref')
        self.robot_radius = config.getfloat('robot', 'radius')
        self.robot_v_pref = config.getfloat('robot', 'v_pref')
        self.robot_visible = config.getboolean('robot', 'visible')
        self._alloc()

    def _alloc(self):
        B = self.B
        # everything a host-side caller reads after a step sits in one slab (see Slab)
        self.out_slab = Slab(host_visible_layout(B, self.human_num), self.device)
        self.state = DeviceState(B, self.human_num, self.device, slab=self.out_slab)
        self.action = torch.zeros((B, 2), dtype=torch.float64, device=self.device)
        self.action_out, self.next_action = self.out_slab['action_out'], self.out_slab['next_action']
        self.reward, self.dmin = self.out_slab['reward'], self.out_slab['dmin']
        self.done, self.info = self.out_slab['done'], self.out_slab['info']
        self.obs32 = self.out_slab['obs32']
        self.write_obs32 = False                 # step() also writes the float32 observation (HostStepper(obs='f32'))
        self._seed32 = torch.zeros(B, dtype=torch.int32, device=self.device)

    def set_robot_policy(self, kind):
        """'orca' / 'linear': the robot decides inside the step kernel (ORCA.predict / Linear.predict of its pre-step state);
        'external_xy' ('holonomic') / 'external_rot' ('unicycle'): step() takes the robot's actions."""
        self.robot_policy = {'orca': _abi.ROBOT_ORCA, 'linear': _abi.ROBOT_LINEAR, 'external_xy': _abi.ROBOT_EXTERNAL_XY,
                             'holonomic': _abi.ROBOT_EXTERNAL_XY, 'external_rot': _abi.ROBOT_EXTERNAL_ROT,
                             'unicycle': _abi.ROBOT_EXTERNAL_ROT}[kind]

    def robot_decides_on_device(self):
        return self.robot_policy in (_abi.ROBOT_ORCA, _abi.ROBOT_LINEAR)

    def params(self):
        return _abi.Params(self.time_step, float(self.time_limit), self.success_reward, self.collision_penalty,
                           self.discomfort_dist, self.discomfort_penalty_factor, self.neighbor_dist, self.time_horizon,
                           self.max_neighbors, self.human_safety_space, self.robot_safety_space,
                           int(bool(self.robot_visible)), self.robot_policy, self.human_policy)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- episodes ------------------------------------------------------------------------------------------------
    def track_episodes(self, k, gamma=0.9):
        self.episodes = EpisodeBuffers(self.B, k, self.device, gamma, self.time_step, self.robot_v_pref,
                                       max_steps=max_episode_steps(self.time_limit, self.time_step))
        return self.episodes

    # ---- reset ---------------------------------------------------------------------------------------------------
    def reset(self, phase='test', cases=None, mask=None, rule=None):
        """Generate scenes on device. `cases` [B] int (tensor/array) are case numbers of `phase`
        (seed = offset[phase] + case, crowd_sim.py:270-276); default: consecutive cases from case_counter[phase]."""
        assert phase in ('train', 'val', 'test')
        if cases is None:
            start = self.case_counter[phase]
            cases = (torch.arange(self.B, dtype=torch.int64) + start) % self.case_size[phase]
            self.case_counter[phase] = int((start + self.B) % self.case_size[phase])
        cases = torch.as_tensor(cases, dtype=torch.int64)
        self.reset_seeds(cases + _PHASE_OFFSET[phase], mask=mask,
                         rule=rule or (self.test_sim if phase == 'test' else self.train_val_sim))
        return self.observation()

    def set_seeds(self, seeds):
        """Load per-slot MT19937 seeds (any integer tensor/array, values in [0, 2**32))."""
        seeds = torch.as_tensor(seeds, dtype=torch.int64).to(self.device, non_blocking=True)
        # uint32 bit patterns stored in an int32 tensor
        self._seed32.copy_(((seeds + 2 ** 31) % 2 ** 32 - 2 ** 31).to(torch.int32))

    def _reset_args(self, mask, rule, seed_stride, use_queue):
        q = use_queue and self._case_counter is not None
        return _abi.ResetArgs(_ptr(mask), _ptr(self._seed32), int(seed_stride) % 2 ** 32, _abi.RULES[rule], self.circle_radius,
                              self.square_width, self.human_radius, self.human_v_pref, self.robot_radius, self.robot_v_pref,
                              self.discomfort_dist, int(bool(self.randomize_attributes)),
                              _ptr(self._case_counter) if q else None, self._case_total if q else 0, self._seed_base if q else 0,
                              self._case_first if q else 0, self._case_wrap if q else 0)

    def reset_seeds(self, seeds=None, mask=None, rule='circle_crossing', seed_stride=0, use_queue=False):
        """crowdsim_reset for the envs selected by `mask` (uint8 device tensor, None = all) from the per-slot seeds.
        With seed_stride != 0 the slot's seed is advanced on device after use; with use_queue the seeds come from the
        shared case queue set up by set_case_queue()."""
        if seeds is not None:
            self.set_seeds(seeds)
        if mask is not None and not (isinstance(mask, torch.Tensor) and mask.dtype == torch.uint8 and mask.device == self.device):
            mask = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8)
        a = self._reset_args(mask, rule, seed_stride, use_queue)
        st = self.state.struct()
        ep = self.episodes.struct() if self.episodes is not None else None
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_reset(C.byref(a), self.B, self.human_num, C.byref(st),
                                         C.byref(ep) if ep is not None else None, self._stream())
        _abi.check(rc, 'crowdsim_reset')
        self._keep = (mask, a)

    # ---- auto-reset with prefetched scenes -------------------------------------------------------------------------
    def set_case_queue(self, first_case, total, phase='test'):
        """Shared work queue of `total` cases starting at `first_case` of `phase` (seed = offset[phase] + case):
        env slots pull the next case on device when their episode ends (Explorer.run_k_episodes with k > slots)."""
        self._case_counter = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._case_total = int(total)
        size = self.case_size[phase] if self.case_size else 0
        if 0 < size < 2 ** 31:
            # the run may cross the end of the phase's case range: case numbers wrap like crowd_sim.py:283 does
            self._seed_base, self._case_first, self._case_wrap = _PHASE_OFFSET[phase], int(first_case) % size, size
        else:                                                # train: 2**32 - 2001 cases, no wrap within int32 counters
            self._seed_base, self._case_first, self._case_wrap = (_PHASE_OFFSET[phase] + int(first_case)) % 2 ** 32, 0, 0

    def enable_autoreset(self, rule='circle_crossing', seed_stride=0):
        """Allocate the per-slot next-scene buffers; step() then re-initialises finished envs in the same launch.
        Call prefetch() (any stream) to (re)fill consumed slots."""
        self.autoreset = AutoResetBuffers(self.B, self.human_num, self.device, self.circle_radius, self.robot_radius,
                                          self.robot_v_pref)
        self._ar_rule, self._ar_seed_stride = rule, seed_stride
        return self.autoreset

    def prefetch(self):
        a = self._reset_args(None, self._ar_rule, self._ar_seed_stride, True)
        ar = self.autoreset.struct()
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_prefetch_scenes(C.byref(a), self.B, self.human_num, C.byref(ar), self._stream())
        _abi.check(rc, 'crowdsim_prefetch_scenes')

    # ---- step ----------------------------------------------------------------------------------------------------
    def step(self, actions=None, n_steps=1):
        """One lockstep env-step. `actions` [B][2] float64 device tensor (vx,vy) / (v,r); None when the robot runs ORCA or
        Linear. n_steps > 1: crowdsim_step_n -- exactly n_steps single steps; with an ORCA / Linear robot and N <= 5 they run inside ONE
        kernel launch with the state in registers (the closed episode loop of explorer.py:41-43). The returned reward /
        done / info are those of each env's last live step."""
        if not self.robot_decides_on_device():
            if actions is None:
                raise ValueError('robot policy is external: actions required')
            if actions.data_ptr() != self.action.data_ptr():
                self.action.copy_(actions, non_blocking=True)
        prm = self.params()
        st = self.state.struct()
        io = _abi.StepIO(_ptr(self.action), _ptr(self.action_out), _ptr(self.reward), _ptr(self.dmin),
                         _ptr(self.done), _ptr(self.info), _ptr(self.obs32) if self.write_obs32 else None)
        ep = self.episodes.struct() if self.episodes is not None else None
        ar = self.autoreset.struct() if self.autoreset is not None else None
        if n_steps == 1:
            with torch.cuda.device(self.device):
                rc = self.lib.crowdsim_step(C.byref(prm), self.B, self.human_num, C.byref(st), C.byref(io),
                                            C.byref(ep) if ep is not None else None, C.byref(ar) if ar is not None else None,
                                            self._stream())
        else:
            with torch.cuda.device(self.device):
                rc = self.lib.crowdsim_step_n(C.byref(prm), self.B, self.human_num, C.byref(st), C.byref(io),
                                              C.byref(ep) if ep is not None else None, C.byref(ar) if ar is not None else None,
                                              int(n_steps), self._stream())
        _abi.check(rc, 'crowdsim_step')
        return self.observation(), self.reward, self.done, self.info

    def step_n(self, n_steps):
        """n_steps closed-loop env-steps (ORCA or Linear robot): see step()."""
        return self.step(None, n_steps=n_steps)

    def orca_act(self, out=None):
        out = self.action_out if out is None else out
        prm = self.params(); st = self.state.struct()
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_orca_act(C.byref(prm), self.B, self.human_num, C.byref(st), _ptr(out), self._stream())
        _abi.check(rc, 'crowdsim_orca_act')
        return out

    def observation(self):
        """[B][N][5] view material: (px, py, vx, vy, radius) of each human (agent.py:60-61), as separate tensors."""
        s = self.state
        return s.h_pos, s.h_vel, s.h_attr[..., 0]

    # ---- value-network support -----------------------------------------------------------------------------------
    def pack_joint(self, unicycle=False, out=None):
        if out is None:
            out = torch.empty((self.B, self.human_num, 13), dtype=torch.float32, device=self.device)
        st = self.state.struct()
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_pack_joint(self.B, self.human_num, C.byref(st), int(unicycle), _ptr(out), self._stream())
        _abi.check(rc, 'crowdsim_pack_joint')
        return out

    def lookahead_pack(self, actions, unicycle=False, out_states=None, out_reward=None):
        """actions [A][2] float64 device tensor -> (states [B][A][N][13] f32, reward [B][A] f64)."""
        A = actions.shape[0]
        if out_states is None:
            out_states = torch.empty((self.B, A, self.human_num, 13), dtype=torch.float32, device=self.device)
        if out_reward is None:
            out_reward = torch.empty((self.B, A), dtype=torch.float64, device=self.device)
        prm = self.params(); st = self.state.struct()
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_lookahead_pack(C.byref(prm), self.B, self.human_num, C.byref(st), _ptr(actions), A,
                                                  int(unicycle), _ptr(out_states), _ptr(out_reward), self._stream())
        _abi.check(rc, 'crowdsim_lookahead_pack')
        return out_states, out_reward


    def human_counts(self):
        """Humans present per env [B] (int64). Differs from human_num only for scenes of rule `mixed` (crowd_sim.py:103-151),
        whose unused human slots are parked at x >= CROWDSIM_PARKED_X (include/crowdsim_b200.h)."""
        return (self.state.h_pos[:, :, 0] < _abi.PARKED_X / 2).sum(dim=1)

    def lookahead_humans(self, out_pos=None, out_vel=None):
        """The observation of env.onestep_lookahead (crowd_sim.py:414-416): the humans' next positions / velocities
        [B][N][2] float64 under their own ORCA decisions; the state is not touched."""
        if out_pos is None:
            out_pos = torch.empty((self.B, self.human_num, 2), dtype=torch.float64, device=self.device)
        if out_vel is None:
            out_vel = torch.empty((self.B, self.human_num, 2), dtype=torch.float64, device=self.device)
        prm = self.params(); st = self.state.struct()
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_lookahead_humans(C.byref(prm), self.B, self.human_num, C.byref(st), _ptr(out_pos), _ptr(out_vel),
                                                    self._stream())
        _abi.check(rc, 'crowdsim_lookahead_humans')
        return out_pos, out_vel

    def onestep_lookahead(self, actions, out_pos=None, out_vel=None):
        """env.onestep_lookahead for one action per env ([B][2] float64 device tensor): ((next_h_pos, next_h_vel, radius),
        reward, done, info) like step(), nothing mutated (crowdsim_onestep_lookahead)."""
        B, N = self.B, self.human_num
        out_pos = torch.empty((B, N, 2), dtype=torch.float64, device=self.device) if out_pos is None else out_pos
        out_vel = torch.empty((B, N, 2), dtype=torch.float64, device=self.device) if out_vel is None else out_vel
        if actions.data_ptr() != self.action.data_ptr():
            self.action.copy_(actions, non_blocking=True)
        prm = self.params(); st = self.state.struct()
        io = _abi.StepIO(_ptr(self.action), _ptr(self.action_out), _ptr(self.reward), _ptr(self.dmin), _ptr(self.done), _ptr(self.info), None)
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_onestep_lookahead(C.byref(prm), B, N, C.byref(st), C.byref(io), _ptr(out_pos), _ptr(out_vel), self._stream())
        _abi.check(rc, 'crowdsim_onestep_lookahead')
        return (out_pos, out_vel, self.state.h_attr[..., 0]), self.reward, self.done, self.info

    def human_times(self, human_times=None, max_steps=4000):
        """CrowdSim.get_human_times for every env (crowdsim_human_times): (human_times [B][N], global_time [B], final
        positions [B][N+1][2] robot first). `human_times`: arrivals recorded during the episode (0 = not yet)."""
        B, N = self.B, self.human_num
        ht = torch.zeros((B, N), dtype=torch.float64, device=self.device) if human_times is None else human_times.to(self.device, torch.float64).contiguous()
        gt = torch.empty((B,), dtype=torch.float64, device=self.device)
        fp = torch.empty((B, N + 1, 2), dtype=torch.float64, device=self.device)
        prm = self.params(); st = self.state.struct()
        # the centralised simulation has its own constants (neighborDist, maxNeighbors, timeHorizon = 10, 10, 5;
        # crowd_sim.py:220), whatever the env's ORCA agents use
        prm.neighbor_dist, prm.max_neighbors, prm.time_horizon = 10.0, 10, 5.0
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_human_times(C.byref(prm), B, N, C.byref(st), _ptr(ht), _ptr(gt), _ptr(fp), int(max_steps), self._stream())
        _abi.check(rc, 'crowdsim_human_times')
        return ht, gt, fp

    def occupancy_maps(self, h_pos=None, h_vel=None, cell_num=4, cell_size=1.0, om_channel_size=3, out=None):
        """MultiHumanRL.build_occupancy_maps (multi_human_rl.py:109-163) for every env: [B][N][cell_num^2 * channels]
        float32. Default input = the live human state; pass the output of lookahead_humans() for next-state maps."""
        if self.human_num < 2:
            raise ValueError('need at least one array to concatenate')      # what the reference's np.concatenate raises
        h_pos = self.state.h_pos if h_pos is None else h_pos
        h_vel = self.state.h_vel if h_vel is None else h_vel
        if out is None:
            out = torch.empty((self.B, self.human_num, cell_num * cell_num * om_channel_size), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.crowdsim_occupancy_maps(self.B, self.human_num, _ptr(h_pos), _ptr(h_vel), int(cell_num), float(cell_size),
                                                  int(om_channel_size), _ptr(out), self._stream())
        _abi.check(rc, 'crowdsim_occupancy_maps')
        return out


class HostStepper(object):
    """env.step() for callers that live on the host (the reference's calling convention: the policy hands a robot
    action to env.step and gets observation, reward, done, info back -- crowd_nav/utils/explorer.py:42-43).

    One call = one CUDA graph replay: H2D copy of the robot actions from pinned memory, the fused step kernel, a refill of
    the consumed next-scene slots on a side branch (when env.enable_autoreset() was called), the robot's next ORCA
    decision (optional, so a host loop can drive an ORCA robot), ONE D2H copy of the slab range holding what the caller
    reads, then a stream synchronise.
    obs = 'f32' (default): the observation comes down as float32 (px, py, vx, vy) per human -- crowdsim_step_io.obs32, the
    cast the reference's value-network policies apply anyway (multi_human_rl.py:43) -- 114 B per env and step at N = 5;
    obs = 'f64': the float64 state arrays themselves, 210 B per env.
    Buffers: self.h_action [B][2] (write before step()); results as views of the pinned host slab: self.h_obs32 [B][N][4]
    (obs = 'f32') or self.h_pos, h_vel [B][N][2] (obs = 'f64'), h_reward, h_dmin, h_done, h_info [B], h_next_action [B][2]
    (.numpy() views are free).
    transfer = 'copy' (default): the buffers cross the link with copy-engine transfers (one up, one down per step).
    transfer = 'direct': the kernels read the action from, and write the step's results to, the pinned host buffers
    themselves (unified addressing: the same pointers are valid on the device) -- the same bytes cross the link on every
    step, but as loads / stores of the step and decision kernels instead of two DMA transfers with their fixed set-up cost;
    the results are visible to the host once the step's event has completed (wait())."""

    def __init__(self, env, next_orca_action=True, obs='f32', prefetch_every=4, transfer='copy'):
        assert obs in ('f32', 'f64') and transfer in ('copy', 'direct')
        assert transfer == 'copy' or obs == 'f32', "transfer='direct' serves the float32 observation"
        self.env, self.obs, self.transfer = env, obs, transfer
        B, N, dev = env.B, env.human_num, env.device
        self.h_action = torch.zeros((B, 2), dtype=torch.float64).pin_memory()
        self.host_slab = Slab(host_visible_layout(B, N), 'cpu', pin=True)
        hs = self.host_slab
        self.h_obs32, self.h_pos, self.h_vel, self.h_reward, self.h_dmin = hs['obs32'], hs['h_pos'], hs['h_vel'], hs['reward'], hs['dmin']
        self.h_done, self.h_info, self.h_action_out, self.h_next_action = hs['done'], hs['info'], hs['action_out'], hs['next_action']
        self.stream = torch.cuda.Stream(device=dev)
        self.side = torch.cuda.Stream(device=dev)
        self.done_event = torch.cuda.Event()
        env.write_obs32 = (obs == 'f32')
        if obs == 'f32':
            lo, hi = 0, (hs.offsets['next_action'][0] + hs.offsets['next_action'][1]) if next_orca_action else (hs.offsets['info'][0] + hs.offsets['info'][1])
        else:
            lo, hi = hs.offsets['reward'][0], hs.offsets['h_vel'][0] + hs.offsets['h_vel'][1]
        self.h2d_bytes = self.h_action.numel() * 8
        self.d2h_bytes = hi - lo
        if transfer == 'direct':                      # what the kernels store to host memory per step
            self.d2h_bytes = B * (N * 16 + 8 + 8 + 1 + 1 + (16 if next_orca_action else 0))
        self.kernels_per_step = 1 + (1 if env.autoreset is not None else 0) + (1 if next_orca_action else 0)

        # The refill of the consumed next-scene slots only has to come round before the same slot's NEXT episode ends, and
        # an episode lasts at least ~7 steps: a refill launch on every prefetch_every-th step (default 4) loses nothing, while
        # one per step keeps 32 blocks x 78 KB of shared memory busy for ~76 us on every step of every batch in flight.
        self.prefetch_every = max(1, int(prefetch_every))
        self._n_launched = 0

        direct = transfer == 'direct'
        if direct:
            # the env's per-step inputs / outputs now ARE the pinned host buffers (device-visible through unified addressing)
            env.action, env.obs32, env.reward, env.dmin = self.h_action, self.h_obs32, self.h_reward, self.h_dmin
            env.done, env.info, env.next_action, env.action_out = self.h_done, self.h_info, self.h_next_action, None

        def body(with_refill=True):
            if not direct:
                env.action.copy_(self.h_action, non_blocking=True)
            env.step(env.action)                       # installs prefetched scenes of finished envs when auto-reset is on
            if env.autoreset is not None and with_refill:   # refill consumed slots on a side branch of the graph
                self.side.wait_stream(self.stream)
                with torch.cuda.stream(self.side):
                    env.prefetch()
            # ONE device->host copy. (Splitting it so that the step results go down while the next-decision kernel runs
            # was measured: 47 M vs 54 M env-steps/s -- the extra stream hand-offs cost more than the overlap gains.)
            if next_orca_action:
                env.orca_act(env.next_action)
            if not direct:
                hs.buf[lo:hi].copy_(env.out_slab.buf[lo:hi], non_blocking=True)
            if env.autoreset is not None and with_refill:
                self.stream.wait_stream(self.side)     # join the side branch
        with torch.cuda.stream(self.stream):
            body()                                     # warm-up outside capture (lazy inits)
        self.stream.synchronize(); self.side.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            body()
        self._lib = _abi.load()
        self._exec = self.graph.raw_cuda_graph_exec()
        self._exec_plain = self._exec                  # the step graph without the refill branch
        if env.autoreset is not None and self.prefetch_every > 1:
            self.graph_plain = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_plain, stream=self.stream):
                body(with_refill=False)
            self._exec_plain = self.graph_plain.raw_cuda_graph_exec()
        self.done_event.record(self.stream)            # creates the underlying cudaEvent_t
        self._event_h = self.done_event.cuda_event
        self._stream_h = self.stream.cuda_stream
        self._result = ((self.h_obs32,) if obs == 'f32' else (self.h_pos, self.h_vel), self.h_reward, self.h_done, self.h_info)
        self.np_action, self.np_next_action = self.h_action.numpy(), self.h_next_action.numpy()

    def step(self):
        self.launch()
        return self.wait()

    # Split form of step() for callers that keep several independent env batches in flight (one HostStepper per batch,
    # each with its own streams and pinned buffers): launch() enqueues the step of this batch and returns at once, wait()
    # blocks until its results are in the host buffers. The uploads/downloads of one batch then overlap the kernels of the
    # others; every batch still pays its own H2D action copy and D2H result copy on every step.
    # Both go straight to the library (crowdsim_graph_launch / crowdsim_event_wait on the raw graph-exec, stream and
    # event handles): ~3 us of interpreter time per call instead of ~12 us through torch's stream context + replay().
    def launch(self):
        ex = self._exec if self._n_launched % self.prefetch_every == 0 else self._exec_plain
        self._n_launched += 1
        rc = self._lib.crowdsim_graph_launch(ex, self._stream_h, self._event_h)
        if rc:
            _abi.check(rc, 'crowdsim_graph_launch')

    def wait(self):
        rc = self._lib.crowdsim_event_wait(self._event_h)
        if rc:
            _abi.check(rc, 'crowdsim_event_wait')
        return self._result


class HostStepperGroup(object):
    """Several independent env batches kept in flight from the host, with the round-robin itself in native code
    (crowdsim_host_pump): per batch-step wait for the batch's results, hand the device's next decision back as the action
    (replay mode: h_next_action -> h_action; a caller with its own policy uses HostStepper.launch / wait instead and writes
    h_action itself), enqueue the next step. Every batch-step still pays its H2D action copy and D2H result copy."""

    def __init__(self, steppers, replay_next_action=True):
        self.steppers = list(steppers)
        n = len(self.steppers)
        arr = lambda vals: (C.c_void_p * n)(*vals)  # noqa: E731
        self._execs = arr([s._exec for s in self.steppers])
        self._execs_plain = arr([s._exec_plain for s in self.steppers])
        self._period = self.steppers[0].prefetch_every
        self._round = 0
        self._streams = arr([s._stream_h for s in self.steppers])
        self._events = arr([s._event_h for s in self.steppers])
        self._dst = arr([s.h_action.data_ptr() for s in self.steppers]) if replay_next_action else None
        self._src = arr([s.h_next_action.data_ptr() for s in self.steppers]) if replay_next_action else None
        self._bytes = self.steppers[0].h_action.numel() * 8 if replay_next_action else 0
        self._lib = _abi.load()

    def start(self):
        for s in self.steppers:
            s.launch()

    def run(self, rounds):
        """`rounds` steps of every batch (start() must have been called once); the last steps are left in flight."""
        rc = self._lib.crowdsim_host_pump(len(self.steppers), self._execs, self._execs_plain, self._period, self._round,
                                          self._streams, self._events, self._dst, self._src, self._bytes, int(rounds))
        self._round += int(rounds)
        if rc:
            _abi.check(rc, 'crowdsim_host_pump')

    def wait(self):
        return [s.wait() for s in self.steppers]


def default_config(human_num=5, test_sim='circle_crossing', train_val_sim='circle_crossing', robot_visible=False,
                   randomize_attributes=False, human_policy='orca'):
    """The reference's crowd_nav/configs/env.config:1-37 as a RawConfigParser (values restated, not read from disk)."""
    import configparser
    cfg = configparser.RawConfigParser()
    cfg.read_dict({
        'env': {'time_limit': '25', 'time_step': '0.25', 'val_size': '100', 'test_size': '500',
                'randomize_attributes': 'true' if randomize_attributes else 'false'},
        'reward': {'success_reward': '1', 'collision_penalty': '-0.25', 'discomfort_dist': '0.2',
                   'discomfort_penalty_factor': '0.5'},
        'sim': {'train_val_sim': train_val_sim, 'test_sim': test_sim, 'square_width': '10', 'circle_radius': '4',
                'human_num': str(human_num)},
        'humans': {'visible': 'true', 'policy': human_policy, 'radius': '0.3', 'v_pref': '1', 'sensor': 'coordinates'},
        'robot': {'visible': 'true' if robot_visible else 'false', 'policy': 'none', 'radius': '0.3', 'v_pref': '1',
                  'sensor': 'coordinates'},
    })
    return cfg
