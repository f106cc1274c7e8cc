"""BatchedExplorer: Explorer.run_k_episodes (reference crowd_nav/utils/explorer.py:21-90) over a BatchedCrowdSim.

Same call signature and the same log lines (their format is consumed by crowd_nav/utils/plot.py:38-55, so it is treated
as a wire format), but the k episodes are streamed through the env's B slots on device: a shared case queue hands the
next case number to whichever slot finishes (seed = offset[phase] + case, crowd_sim.py:270-276), scenes are prefetched
on a side stream and installed by the step kernel, per-episode results (terminal class, time, discounted return, danger
statistics) are written by the step kernel into per-case rows. The host only reduces those rows exactly like the
reference does (explorer.py:74-90).

Robot policies:
  'orca'            the robot's ORCA solve is fused into the step kernel (test.py --policy orca)
  'linear'          the robot's Linear.predict is fused into the step kernel (test.py --policy linear)
  a policy object   anything with .act_batch(env) -> [B][2] float64 device tensor of ActionXY (policy.make_sarl() ...)
With update_memory=True the rollout also fills a memory.DeviceReplayMemory like Explorer.update_memory does
(explorer.py:92-125; imitation-learning returns or target-network bootstraps).

Multi-GPU (torchrun, one process per GPU): the k cases are split into contiguous ranges per rank; there is no data-path
collective; ONE gather of the per-case result rows (48 B per episode: 6 float64 columns; NCCL on GPU tensors, gloo in the CPU tests) brings
them to rank 0, which prints the log lines.
"""
import logging

import torch

from . import _abi

INFO_NAMES = {_abi.INFO_REACHGOAL: 'ReachGoal', _abi.INFO_COLLISION: 'Collision', _abi.INFO_TIMEOUT: 'Timeout'}
RESULT_COLS = ('info', 'steps', 'time', 'return', 'too_close', 'min_dist_sum')


def average(input_list):
    """explorer.py:128-132"""
    if input_list:
        return sum(input_list) / len(input_list)
    return 0


def shard_range(k, rank, world):
    """Contiguous block of cases for `rank`: sizes differ by at most one, earlier ranks take the extra ones."""
    base, extra = divmod(k, world)
    start = rank * base + min(rank, extra)
    return start, base + (1 if rank < extra else 0)


def pack_results(ep, n):
    """Per-case result rows of an EpisodeBuffers as one [n][6] float64 tensor (exact for the integer columns)."""
    cols = [ep.res_info[:n].double(), ep.res_steps[:n].double(), ep.res_time[:n], ep.res_return[:n],
            ep.res_too_close[:n].double(), ep.res_min_dist_sum[:n]]
    return torch.stack(cols, dim=1).contiguous()


def gather_results(local_rows, k, rank, world, group=None):
    """The one collective of the path: all ranks' [n_r][6] rows -> [k][6] on every rank, in case order.
    Rows are padded to the largest shard so a single all_gather suffices."""
    if world == 1:
        return local_rows
    import torch.distributed as dist
    n_max = shard_range(k, 0, world)[1]
    pad = torch.zeros((n_max, local_rows.shape[1]), dtype=local_rows.dtype, device=local_rows.device)
    pad[:local_rows.shape[0]] = local_rows
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad, group=group)
    return torch.cat([out[r][:shard_range(k, r, world)[1]] for r in range(world)], dim=0)


def summarize(rows, k, phase, time_limit, time_step, episode=None, print_failure=False, log=logging.info):
    """explorer.py:52-90 on gathered per-case rows ([k][6]: info, steps, time, return, too_close, min_dist_sum).
    Returns the statistics as a dict and emits the reference's log lines through `log`."""
    rows = rows.cpu().tolist()
    success_times, collision_times, timeout_times = [], [], []
    collision_cases, timeout_cases = [], []
    cumulative_rewards = []
    too_close = 0
    min_dist_sum, min_dist_n = 0.0, 0
    for i, (info, steps, t, ret, tc, mds) in enumerate(rows):
        info = int(info)
        if info == _abi.INFO_REACHGOAL:
            success_times.append(t)
        elif info == _abi.INFO_COLLISION:
            collision_cases.append(i); collision_times.append(t)
        elif info == _abi.INFO_TIMEOUT:
            timeout_cases.append(i); timeout_times.append(t)
        else:
            raise ValueError('Invalid end signal from environment')      # explorer.py:64
        cumulative_rewards.append(ret)
        too_close += int(tc); min_dist_sum += mds; min_dist_n += int(tc)
    success, collision, timeout = len(success_times), len(collision_times), len(timeout_times)
    assert success + collision + timeout == k
    success_rate, collision_rate = success / k, collision / k
    avg_nav_time = sum(success_times) / len(success_times) if success_times else time_limit
    extra_info = '' if episode is None else 'in episode {} '.format(episode)
    log('{:<5} {}has success rate: {:.2f}, collision rate: {:.2f}, nav time: {:.2f}, total reward: {:.4f}'.
        format(phase.upper(), extra_info, success_rate, collision_rate, avg_nav_time, average(cumulative_rewards)))
    stats = {'success_rate': success_rate, 'collision_rate': collision_rate, 'timeout_rate': timeout / k,
             'nav_time': avg_nav_time, 'total_reward': average(cumulative_rewards), 'success': success,
             'collision': collision, 'timeout': timeout, 'collision_cases': collision_cases,
             'timeout_cases': timeout_cases, 'env_steps': int(sum(r[1] for r in rows))}
    if phase in ['val', 'test']:
        num_step = sum(success_times + collision_times + timeout_times) / time_step
        avg_min_dist = min_dist_sum / min_dist_n if min_dist_n else 0
        log('Frequency of being in danger: %.2f and average min separate distance in danger: %.2f'
            % (too_close / num_step, avg_min_dist))
        stats['danger_frequency'] = too_close / num_step
        stats['avg_min_dist'] = avg_min_dist
    if print_failure:
        log('Collision cases: ' + ' '.join([str(x) for x in collision_cases]))
        log('Timeout cases: ' + ' '.join([str(x) for x in timeout_cases]))
    return stats


class BatchedExplorer(object):
    def __init__(self, env, robot_policy='orca', device=None, memory=None, gamma=None, target_policy=None,
                 rank=0, world=1, group=None):
        self.env = env
        self.robot_policy = robot_policy
        self.device = device or env.device
        self.memory = memory
        self.gamma = gamma
        self.target_policy = target_policy
        self.target_model = None
        self.rank, self.world, self.group = rank, world, group
        self.last_rows = None
        self.last_env_steps = 0

    def update_target_model(self, target_model):
        import copy
        self.target_model = copy.deepcopy(target_model)

    def run_k_episodes(self, k, phase, update_memory=False, imitation_learning=False, episode=None,
                       print_failure=False, prefetch_every=2, check_every=32, steps_per_launch=8):
        env = self.env
        if update_memory and (self.memory is None or self.gamma is None):
            raise ValueError('Memory or gamma value is not set!')            # explorer.py:93-94
        first_case = env.case_counter[phase]
        start, n_local = shard_range(k, self.rank, self.world)
        gamma = self.gamma if self.gamma is not None else 0.9
        ep = env.track_episodes(max(n_local, 1), gamma)
        rule = env.test_sim if phase == 'test' else env.train_val_sim
        env.set_case_queue((first_case + start) % env.case_size[phase], n_local, phase)    # wraps inside the phase like crowd_sim.py:283
        env.enable_autoreset(rule)
        on_device = self.robot_policy in ('orca', 'linear')
        env.set_robot_policy(self.robot_policy if on_device else 'external_xy')
        env.reset_seeds(rule=rule, use_queue=True)
        recorder = None
        if update_memory:
            from .memory import TrajectoryRecorder
            om = getattr(self.robot_policy, 'om', None) if getattr(self.robot_policy, 'with_om', False) else None
            recorder = TrajectoryRecorder(env, self.memory, self.gamma, imitation_learning, self.target_model, om=om)
        side = torch.cuda.Stream(device=env.device)
        main = torch.cuda.current_stream(env.device)
        # an ORCA / Linear robot decides on device: the episode loop of explorer.py:41-43 closes inside the kernel, several
        # steps per launch (crowdsim_step_n); a recorded rollout or a host-side policy needs every step
        chunk = max(1, int(steps_per_launch)) if (on_device and recorder is None) else 1
        if chunk > 1:
            prefetch_every, check_every = 1, max(1, check_every // chunk)
        from .batched import max_episode_steps
        guard = 2 * (max_episode_steps(env.time_limit, env.time_step) + chunk) * (n_local // max(env.B, 1) + 2) // chunk + 16
        it = 0
        while True:
            if it % prefetch_every == 0:
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    env.prefetch()
            if recorder is not None:
                recorder.before_step()
            if on_device:
                env.step(n_steps=chunk)
            else:
                env.step(self.robot_policy.act_batch(env))
            if recorder is not None:
                recorder.after_step()
            it += 1
            if it % check_every == 0 and int(env.state.active.sum()) == 0 and int(env.autoreset.want.sum()) == 0:
                break
            if it > guard:
                raise RuntimeError('rollout did not terminate')
        main.wait_stream(side)
        rows = gather_results(pack_results(ep, n_local), k, self.rank, self.world, self.group)
        env.case_counter[phase] = (first_case + k) % env.case_size[phase]
        env.autoreset = None
        self.last_rows = rows
        if self.rank != 0:
            return None
        stats = summarize(rows, k, phase, env.time_limit, env.time_step, episode, print_failure)
        self.last_env_steps = stats['env_steps']
        return stats
