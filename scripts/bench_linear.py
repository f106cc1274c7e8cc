#!/usr/bin/env python
"""Throughput of the Linear-policy paths on one GPU, by bench.py's steady-state method, next to bench.py itself.

  python scripts/bench_linear.py [--rounds 25] [--no-bench]

Workloads (circle crossing, N = 5, train-phase case queues, auto-reset and scene refill on):
  orca_robot_linear_humans   the robot runs ORCA, the humans Linear
  linear_robot_orca_humans   the robot runs Linear, the humans ORCA
  linear_both                both Linear
Method for each (bench.py's): 64 independent 4096-env batches (state larger than L2), batch p on stream p mod 16, one
crowdsim_step_n(16) launch per batch per round, the refill of consumed next-scene slots on a side stream; >= 384 env-steps
of warm-up per env, then --rounds rounds between two CUDA events; value = env-steps performed / elapsed time.
Plus square20_linear_humans: one 4096-env x N = 20 square-crossing crowd-kernel launch (crowdsim_step) with linear humans,
and the same launch with ORCA humans, CUDA events around 200 back-to-back launches each.
The same call runs `python bench.py --gpus 1` (ORCA humans) and reads the GPU's name and power limit. Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else 'unknown (%s)' % out.stderr.strip()


def steady_state(robot, humans, rounds, B=4096, pools=64, S=16, C=16, N=5, rule='circle_crossing'):
    import torch
    from crowdnav_b200 import _abi
    from crowdnav_b200.batched import BatchedCrowdSim, default_config
    lib = _abi.load()
    warm = -(-384 // C)
    envs = []
    for p in range(pools):
        env = BatchedCrowdSim(B)
        env.configure(default_config(human_num=N, test_sim=rule, train_val_sim=rule, human_policy=humans))
        env.set_robot_policy(robot)
        env.k_total = B * ((warm + rounds + 8) * C // 3 + 4)          # episodes last >= 3 steps (a linear robot collides early)
        env.track_episodes(env.k_total, gamma=0.9)
        env.set_case_queue(p * env.k_total, env.k_total, 'train')
        env.enable_autoreset(rule)
        env.reset_seeds(rule=rule, use_queue=True)
        env.prefetch()
        envs.append(env)
    lanes = [torch.cuda.Stream() for _ in range(S)]
    sides = [torch.cuda.Stream() for _ in range(S)]
    for s in range(S):
        with torch.cuda.stream(lanes[s]):
            envs[s].step_n(C); envs[s].prefetch()
    torch.cuda.synchronize()

    def graph(s, fn, side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=sides[s] if side else lanes[s]):
            for p in range(s, pools, S):
                fn(envs[p])
        return g
    graphs = [graph(s, lambda e: e.step_n(C), False) for s in range(S)] + [graph(s, lambda e: e.prefetch(), True) for s in range(S)]
    execs = [(g.raw_cuda_graph_exec(), (lanes + sides)[i].cuda_stream) for i, g in enumerate(graphs)]
    main = torch.cuda.current_stream()

    def run(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for ls in lanes + sides:
            ls.wait_event(e0)
        for _ in range(n):
            for ex, sh in execs:
                _abi.check(lib.crowdsim_graph_launch(ex, sh, None), 'crowdsim_graph_launch')
        for ls in lanes + sides:
            ev = torch.cuda.Event(); ev.record(ls); main.wait_event(ev)
        e1.record(main)
        return e0, e1

    def done():
        tot = 0
        for env in envs:
            n = int(min(env._case_counter.item(), env.k_total))
            tot += int(env.episodes.res_steps[:n].sum().item()) + int((env.episodes.ep_steps * env.state.active.to(torch.int32)).sum().item())
        return tot
    run(warm)
    torch.cuda.synchronize()
    before = done()
    e0, e1 = run(rounds)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    steps = done() - before
    return {'robot': robot, 'humans': humans, 'N': N, 'value': steps / (ms * 1e-3), 'unit': 'env-steps/s', 'ms': ms,
            'env_steps': steps, 'env_steps_launched': pools * B * C * rounds, 'batches': pools, 'envs_per_batch': B,
            'streams': S, 'steps_per_launch': C, 'warmup_env_steps': warm * C}


def crowd_launch(humans, B=4096, N=20, reps=200):
    import torch
    from crowdnav_b200.batched import BatchedCrowdSim, default_config
    env = BatchedCrowdSim(B)
    env.configure(default_config(human_num=N, test_sim='square_crossing', train_val_sim='square_crossing', human_policy=humans))
    env.set_robot_policy('orca')
    env.reset('train', rule='square_crossing')
    for _ in range(20):
        env.step()
    env.state.g_time.zero_()                    # mid-episode crowds; finished envs keep stepping (no bookkeeping in this leg)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        env.step()
    e1.record()
    torch.cuda.synchronize()
    us = 1e3 * e0.elapsed_time(e1) / reps
    return {'humans': humans, 'N': N, 'rule': 'square_crossing', 'envs': B, 'us_per_launch': us, 'env_steps_per_s': B / (us * 1e-6),
            'launches': reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=25)
    ap.add_argument('--no-bench', action='store_true')
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'bench_linear.py measures on a GPU'
    out = {'gpu': gpu_info(), 'workloads': {}}
    for name, robot, humans in (('orca_robot_linear_humans', 'orca', 'linear'), ('linear_robot_orca_humans', 'linear', 'orca'),
                                ('linear_both', 'linear', 'linear')):
        out['workloads'][name] = steady_state(robot, humans, args.rounds)
        torch.cuda.empty_cache()
    out['workloads']['square20_linear_humans'] = crowd_launch('linear')
    out['workloads']['square20_orca_humans'] = crowd_launch('orca')
    if not args.no_bench:
        b = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1'], capture_output=True, text=True, cwd=ROOT)
        lines = [l for l in b.stdout.strip().splitlines() if l.startswith('{')]
        out['bench_py_orca_humans'] = json.loads(lines[-1]) if lines else {'error': b.stderr[-2000:]}
    print(json.dumps(out))


if __name__ == '__main__':
    main()
