#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched CrowdSim-v0 step path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs 4096] [--humans 5] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] = 4096 batched envs x 5 ORCA humans, circle_crossing, ORCA robot,
robot invisible, per GPU. Because 4096 envs of state are only 2.6 MB, the bench holds POOLS independent batches whose
combined state exceeds the 126 MB L2 ("inputs larger than L2"). One bench "step" = one call of the hot path on every
batch: crowdsim_step_n advances each env by C env-steps (--chunk, default 16) in one launch of the fused step kernel (6
ORCA solves/env, collision/reward/terminal, integration, episode bookkeeping), and one scene-prefetch launch per batch on
a side stream re-generates the scenes of envs whose episode ended (fresh MT19937 seeds), so every env is live on every
env-step. The timed region is exactly K such steps; batch p always runs on stream p mod S (--streams, default 16), so the
steps of one batch stay ordered while independent batches overlap on the device. `value` = env-steps PERFORMED (counted by the step kernel) / device time;
`single_stream` = the same with one batch in flight; `e2e` = HostStepper.launch()/wait() over 16 batches with pinned host
buffers in and out on every batch-step; `roofline` = the step kernel alone (single-stream graph, CUDA events).

Printed JSON keys follow the driver contract; see DESIGN.md "Measurement" for definitions. The oracle (oracle/) is
executed here ONLY in the cpu_baseline leg and in --impl reference.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

try:                                             # the metric string is BASELINE.json's, verbatim
    with open(os.path.join(ROOT, 'BASELINE.json')) as _f:
        METRIC = json.load(_f)['metric']
except Exception:
    METRIC = 'env-steps/sec at 5 humans x batched envs; 500-case success/collision parity'
ALG_BYTES = lambda n: 8 * (19 + 12 * n) + 2      # SURVEY.md 8(d): 634 B at N=5, 2074 B at N=20  # noqa: E731


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=25, help='timed steps; one step advances every env on the GPU by --chunk env-steps')
    ap.add_argument('--warmup', type=int, default=24, help='steps before the timed region (at least 384 env-steps per env: a steady mix of episode phases)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--envs', type=int, default=4096, help='envs per batch per GPU')
    ap.add_argument('--humans', type=int, default=5)
    ap.add_argument('--pools', type=int, default=0, help='independent batches rotated through (0 = enough to exceed L2)')
    ap.add_argument('--rule', default='circle_crossing')
    ap.add_argument('--streams', type=int, default=16, help='independent env batches stepped concurrently (CUDA streams inside the timed graph)')
    ap.add_argument('--e2e-batches', type=int, default=16, help='independent env batches kept in flight by the e2e leg')
    ap.add_argument('--e2e-obs', default='f32', choices=['f32', 'f64'], help='observation format of the e2e leg (HostStepper obs=)')
    ap.add_argument('--e2e-transfer', default='auto', choices=['auto', 'direct', 'copy'], help="how the e2e leg's host buffers cross the link: the kernels load / store pinned host memory themselves (better for 4096-env batches: 3.0e8 vs 2.8e8), or copy-engine transfers (better for 16384-env batches: 3.96e8 vs 3.6e8 per GPU); auto = by the bytes per step")
    ap.add_argument('--chunk', type=int, default=16, help='env-steps per launch (crowdsim_step_n); 1 = one launch per step. 8 / 12 / 16 / 24 give 839 / 866 / 905 / 883 M env-steps/s (24: 6 %% of the env-steps lost to envs waiting for a scene refill)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-python-loop', action='store_true', help='reference arm: skip the reference-shaped Python loop timing')
    ap.add_argument('--no-scale', action='store_true', help='skip the supplementary 1 Mi-env launch measurement')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write a seeded sample of the per-case episode '
                    'rows the timed path recorded as DIR/<name>.npy (float64), for comparing two builds output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be >= 1')
    return args


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(object):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe): one long-lived
    `nvidia-smi -lms 20` child whose lines are timestamped on arrival; only samples that fall between mark_start() and
    mark_stop() are used (the child is started earlier so that its start-up cost is outside the window)."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.rows, self.t0, self.t1 = [], None, None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        if self.proc is None:
            return
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(',')]))

    def wait_ready(self, timeout=20.0):
        """Block until the child has delivered its first sample (nvidia-smi can take seconds to start on a cold box)."""
        t_end = time.perf_counter() + timeout
        while not self.rows and time.perf_counter() < t_end and self.proc is not None and self.proc.poll() is None:
            time.sleep(0.01)
        return bool(self.rows)

    def mark_start(self):
        self.t0 = time.perf_counter()

    def mark_stop(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()            # the child we started, by handle
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        self.thread.join(timeout=5)
        inside = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or 1e30) and len(r) >= 7]
        used = inside if inside else [r for _, r in self.rows[-3:] if len(r) >= 7]
        num = lambda v: int(float(v)) if v.replace('.', '', 1).isdigit() else None  # noqa: E731
        sm = sorted(x for x in (num(r[0]) for r in used) if x is not None)
        mx = [x for x in (num(r[1]) for r in used) if x is not None]
        pw = [float(r[2]) for r in used if r[2].replace('.', '', 1).isdigit()]
        reasons = set()
        for r in used:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(inside), 'power_w_max': max(pw) if pw else None,
                'note': None if inside else 'timed region shorter than the sampling period: nearest samples used'}


# ----------------------------------------------------------------------------------------------------------------------
def usable_cpus():
    """Logical CPUs this process may run on (cgroup / affinity mask aware), not os.cpu_count()."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


class CpuArm(object):
    """The CPU arm: the C restatement of the reference loop (oracle/crowdsim_oracle.c), one batch of `envs` envs stepped in
    lockstep inside ONE OpenMP parallel region (every thread owns a fixed range of envs, one barrier per pass, finished envs
    are re-seeded in place). 'All the host threads it can use' is calibrated, because a barrier per 270 us pass collapses
    when the region is oversubscribed: every candidate thread count (usable CPUs, /2, /4, ...) is timed over windows of
    >= 0.4 s and the best median wins; the timed run is then checked against the calibrated rate."""

    def __init__(self, args):
        import numpy as np
        sys.path.insert(0, os.path.join(ROOT, 'oracle'))
        os.environ.setdefault('OMP_WAIT_POLICY', 'passive')      # before libgomp starts: spinning waiters make oversubscription fatal
        os.environ.setdefault('OMP_PROC_BIND', 'false')
        import pyoracle as po
        self.po, self.np, self.args = po, np, args
        self.B, self.N = args.envs, args.humans
        self.prm = po.default_params()
        self.st = po.HostState(self.B, self.N); self.io = po.HostStepIO(self.B)
        self.seeds = (np.arange(self.B) + 2000).astype(np.uint32)
        po.reset(self.st, self.seeds, args.rule, seed_stride=self.B)
        self.passes(60)                                          # into steady state (episodes at all phases)
        self.calibration = {}

    def passes(self, n):
        self.po.run_passes(self.prm, self.st, self.io, self.seeds, n, self.args.rule, seed_stride=self.B)

    def rate(self, seconds, block=20):
        """env-steps/s over a window of >= `seconds`."""
        t0 = time.perf_counter(); n = 0
        while time.perf_counter() - t0 < seconds:
            self.passes(block); n += block
        return n * self.B / (time.perf_counter() - t0)

    def calibrate(self):
        n = usable_cpus()
        cands = sorted({max(1, n >> s) for s in range(0, 6)}, reverse=True)
        best = (0.0, 1)
        for th in cands:
            self.po.set_threads(th)
            self.passes(5)
            r = sorted(self.rate(0.4) for _ in range(3))[1]      # median of three 0.4 s windows
            self.calibration[th] = r
            if r > best[0]:
                best = (r, th)
            if r < 0.5 * best[0] and th < best[1]:               # past the optimum: fewer threads only get slower
                break
        self.threads, self.calibrated_rate = best[1], best[0]
        self.po.set_threads(self.threads)
        return self.threads

    def timed(self, steps, warmup, min_seconds=1.0):
        """`steps` lockstep passes per replay, replays back to back for >= min_seconds: returns (median replay seconds,
        replays, min, max). If the run falls below half the calibrated rate (the host got busy), calibrate again once."""
        for attempt in range(2):
            self.passes(max(warmup, 3))
            ts = []
            t_begin = time.perf_counter()
            while (time.perf_counter() - t_begin < min_seconds or len(ts) < 5) and len(ts) < 20000:
                t0 = time.perf_counter(); self.passes(steps); ts.append(time.perf_counter() - t0)
            ts.sort()
            med = ts[len(ts) // 2]
            if self.B * steps / med >= 0.5 * self.calibrated_rate or attempt == 1:
                return med, len(ts), ts[0], ts[-1], attempt
            self.calibrate()


WORKLOAD = '%d batched envs x %d ORCA humans, %s, ORCA robot (invisible), auto-reset, per GPU'


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = oracle port (the reference is Python + an
    absent native rvo2; it cannot travel to the GPU box), all host threads, same config/metric."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    arm = CpuArm(args)
    cores = arm.calibrate()
    B, N = args.envs, args.humans
    med, replays, tmin, tmax, recal = arm.timed(args.steps, args.warmup, min_seconds=2.0)
    v = B * args.steps / med
    po, prm, st, io, seeds = arm.po, arm.prm, arm.st, arm.io, arm.seeds
    # the same port driven one call per pass from the interpreter (step; reset of the finished envs), like a host loop would
    t1 = time.perf_counter(); n_calls = 0
    while time.perf_counter() - t1 < 1.0:
        po.step(prm, st, io)
        po.reset(st, seeds, args.rule, mask=io.done, seed_stride=B)
        n_calls += 1
    per_call = B * n_calls / (time.perf_counter() - t1)
    # context: the same path with the reference's STRUCTURE (interpreter-bound Python loop around a native rvo2 step,
    # oracle/pyloop.py) on a bounded sample -- the reference's real files cannot travel to this box
    py = None
    if not args.no_python_loop:
        import pyloop
        procs = min(usable_cpus(), 64)
        one, n1 = pyloop.timed_rate(list(range(1000, 1064)), N, args.rule)
        allc, n2, procs = pyloop.timed_rate_all_cores(list(range(1000, 1000 + 16 * procs)), N, args.rule, procs=procs)
        py = {'one_core_env_steps_per_s': one, 'all_cores_env_steps_per_s': allc, 'processes': procs,
              'sample': '%d + %d env-steps of the seeded test cases; Python loop + C rvo2 shim (oracle/pyloop.py); the reference\'s '
                        'own Python measured 4.8 k env-steps/s/core in the build container (DESIGN.md 6)' % (n1, n2)}
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * med / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64 state + f32 ORCA solver', 'data': 'synthetic',
            'config': {'workload': WORKLOAD % (B, N, args.rule), 'envs_per_gpu': B, 'humans': N,
                       'note': 'CPU arm: one %d-env batch stepped in lockstep by all host threads (rank 0 only)' % B},
            'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
                             'sample': 'median of %d back-to-back replays of %d lockstep passes over a %d-env batch (one C call per replay, min %.3g s, max %.3g s); '
                                       'C restatement of the reference loop (oracle/crowdsim_oracle.c, OpenMP: every thread owns a range of envs; '
                                       'thread count calibrated over %s usable CPUs)' % (replays, args.steps, B, tmin, tmax, usable_cpus()),
                             'calibration_env_steps_per_s': {str(k): arm.calibration[k] for k in sorted(arm.calibration)},
                             'recalibrated': bool(recal), 'per_pass_calls_value': per_call},
            'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'python_loop': py, 'gpu_launches': 0}
    print(json.dumps(line))


def cpu_oracle_rate(args, seconds=10.0):
    """cpu_baseline leg of the default run: same arm, `seconds` of CPU work."""
    arm = CpuArm(args)
    cores = arm.calibrate()
    rates = sorted(arm.rate(seconds / 5, block=50) for _ in range(5))
    return rates[2], cores, 'lockstep passes over a %d-env batch (auto-reset) inside one OpenMP region, %.0f s, median of 5 segments (min %.2e, max %.2e); threads calibrated over %d usable CPUs' % (
        args.envs, seconds, rates[0], rates[-1], usable_cpus())


# ----------------------------------------------------------------------------------------------------------------------
DUMP_ROWS = 16384


def dump_episode_rows(out_dir, envs, B):
    """--dump-outputs: the per-case episode rows the step kernel of the timed path recorded (what Explorer.run_k_episodes
    hands its caller: terminal info, steps, time, discounted return, danger count, min-distance sum, final robot position),
    for a fixed seeded sample of DUMP_ROWS of the first 2 x B cases of every batch (claimed by the initial reset and the
    first scene prefetch). A row depends only on its case's seed, not on which env slot ran the case or when, so with the
    same arguments the files are identical from run to run; the slot-level state after the last step is not, because the
    scene refills race the steps by design. Those cases have all ended: an episode lasts at most ~100 steps and the
    warm-up alone is 384."""
    import numpy as np
    import torch
    rng = np.random.RandomState(0)
    per = max(1, DUMP_ROWS // len(envs))
    cols = {k: [] for k in ('seed', 'info', 'steps', 'time', 'return', 'too_close', 'min_dist_sum', 'final_robot_pos')}
    for env in envs:
        idx = torch.from_numpy(np.sort(rng.choice(2 * B, min(per, 2 * B), replace=False))).to(env.device)
        ep = env.episodes
        if not bool((ep.res_steps[idx] > 0).all()):
            raise RuntimeError('--dump-outputs: a sampled case has not ended')
        cols['seed'].append((idx + env._seed_base).double())          # MT19937 seed of the case (train phase: 2000 + case)
        for k, a in (('info', ep.res_info), ('steps', ep.res_steps), ('time', ep.res_time), ('return', ep.res_return),
                     ('too_close', ep.res_too_close), ('min_dist_sum', ep.res_min_dist_sum), ('final_robot_pos', ep.res_final_rpos)):
            cols[k].append(a[idx].double())
    os.makedirs(out_dir, exist_ok=True)
    for k, parts in cols.items():
        np.save(os.path.join(out_dir, 'episode_%s.npy' % k), torch.cat(parts).cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from crowdnav_b200 import _abi
    from crowdnav_b200.batched import BatchedCrowdSim, default_config

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    sampler = ClockSampler(local)                            # started early: its start-up must be over before the timed region
    lib = _abi.load()
    B, N, K, W, C = args.envs, args.humans, args.steps, args.warmup, max(1, args.chunk)
    bytes_per_env = ALG_BYTES(N)
    pools = args.pools or max(2, int(1.3 * 126e6 / (B * bytes_per_env)) + 1)
    S = max(1, min(args.streams, pools))
    pools = (pools + S - 1) // S * S                         # every stream owns the same number of batches

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the timed region: exactly K rounds (every batch advanced by C env-steps in one launch), no gap between them; the
    # streams are only joined at the two ends of the region ----
    rounds = K
    warm_rounds = max(W, -(-384 // C))                       # >= 384 env-steps per env: steady episode mix

    envs = []
    for p in range(pools):
        env = BatchedCrowdSim(B, device=dev)
        env.configure(default_config(human_num=N, test_sim=args.rule, train_val_sim=args.rule))
        env.set_robot_policy('orca')
        # every batch streams its own range of train-phase cases (seed = 2000 + case, crowd_sim.py:272-273) through its
        # B slots; per-episode result rows are recorded on device and reduced once at the end (the path's one collective)
        visits = (warm_rounds + rounds + 8) * C + 600 + (8000 if p < max(1, args.e2e_batches) else 0)   # the first batches also serve the single-batch and e2e legs
        env.k_total = B * (visits // 6 + 4)                  # episodes last >= 7 steps
        env.track_episodes(env.k_total, gamma=0.9)
        env.set_case_queue((rank * pools + p) * env.k_total, env.k_total, 'train')
        env.enable_autoreset(args.rule)
        env.reset_seeds(rule=args.rule, use_queue=True)
        env.prefetch()
        envs.append(env)
    torch.cuda.synchronize()

    # ---- one CUDA graph per stream: for each batch the stream owns, C closed-loop env-steps in ONE launch (crowdsim_step_n:
    # state in registers, finished envs install their prefetched next scene inside the launch) and, on the stream's side
    # stream, the refill of the consumed next-scene slots (it may overlap later launches: release/acquire slot hand-over).
    # The streams never wait for each other: batch p always runs on stream p mod S, a round = every stream replays its graph
    # once; Python only issues S raw graph launches per round (crowdsim_graph_launch, ~3 us each) and stays ahead. ----
    main = torch.cuda.Stream(device=dev)
    lanes = [torch.cuda.Stream(device=dev) for _ in range(S)]
    sides = [torch.cuda.Stream(device=dev) for _ in range(S)]

    def stream_graph(s, batch_ids, n_chunks=1, step_fn=None, side=False):
        """A graph that is a plain sequence of launches on ONE stream (no fork / join): lane graphs step, side graphs refill."""
        g = torch.cuda.CUDAGraph()
        st_ = sides[s] if side else lanes[s]
        with torch.cuda.graph(g, stream=st_):
            for _ in range(n_chunks):
                for p in batch_ids:
                    (step_fn or (lambda e: e.step_n(C) if C > 1 else e.step()))(envs[p])
        return g
    for s in range(S):                                       # lazy initialisations outside capture
        with torch.cuda.stream(lanes[s]):
            envs[s].step(); envs[s].prefetch()
    torch.cuda.synchronize()
    refill = lambda e: e.prefetch()  # noqa: E731
    graphs = [stream_graph(s, list(range(s, pools, S))) for s in range(S)]
    fills = [stream_graph(s, list(range(s, pools, S)), step_fn=refill, side=True) for s in range(S)]
    # a round = every lane replays its step graph, every side stream its refill graph. The refills are NOT ordered against
    # the steps (the generator fills whatever slots it finds EMPTY, the step kernel installs whatever it finds READY:
    # release / acquire hand-over per slot), so no stream ever waits for another one.
    execs = [(g.raw_cuda_graph_exec(), lanes[s].cuda_stream) for s, g in enumerate(graphs)] + \
            [(g.raw_cuda_graph_exec(), sides[s].cuda_stream) for s, g in enumerate(fills)]
    launches_per_round = 2 * pools

    def run_rounds(n, tick=None):
        """n rounds on all streams between two events on `main` (returns them); tick: list that receives one event per round
        recorded on stream 0."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for ls in lanes + sides:
            ls.wait_event(e0)
        for r in range(n):
            for ex, sh in execs:
                rc = lib.crowdsim_graph_launch(ex, sh, None)
                if rc:
                    _abi.check(rc, 'crowdsim_graph_launch')
            if tick is not None:
                ev = torch.cuda.Event(enable_timing=True); ev.record(lanes[0]); tick.append(ev)
        for ls in lanes + sides:
            ev = torch.cuda.Event(); ev.record(ls); main.wait_event(ev)
        e1.record(main)
        return e0, e1

    def env_steps_done(which=None):
        """env-steps actually performed so far on this rank (finished episodes + episodes in progress): an env whose next
        scene is not ready when its episode ends is parked until the refill arrives and performs no env-step meanwhile."""
        tot = 0
        for env in (envs if which is None else which):
            n = int(min(env._case_counter.item(), env.k_total))
            tot += int(env.episodes.res_steps[:n].sum().item()) + int((env.episodes.ep_steps * env.state.active.to(torch.int32)).sum().item())
        return tot

    # ---- warm-up: every batch far into steady state (>= 384 env-steps, i.e. several episode lengths: the mix of episode
    # phases is stationary) ----
    run_rounds(warm_rounds)

    barrier()
    steps_before = env_steps_done()
    sampler.wait_ready()
    ticks = []
    sampler.mark_start()
    e0, e1 = run_rounds(rounds, tick=ticks)
    barrier()
    sampler.mark_stop()
    if args.dump_outputs and rank == 0:
        dump_episode_rows(args.dump_outputs, envs, B)
    launches = rounds * launches_per_round
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    live_steps = env_steps_done() - steps_before             # counted on device by the step kernel itself
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    cnt = torch.tensor([live_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_max = float(t.item())
    live_total = int(cnt.item())
    value = live_total / (ms_max * 1e-3)                     # == world * pools * B * C * K / time unless envs were parked
    # distribution over the rounds (stream 0's clock): a steady region has median ~ mean
    rt = sorted(ticks[i].elapsed_time(ticks[i + 1]) for i in range(len(ticks) - 1)) if len(ticks) > 2 else []
    round_stats = None
    if rt:
        med = rt[len(rt) // 2]
        round_stats = {'rounds': rounds, 'env_steps_per_env': C, 'median_ms': med, 'p10_ms': rt[len(rt) // 10], 'p90_ms': rt[(9 * len(rt)) // 10],
                       'median_value': world * pools * B * C / (med * 1e-3),
                       'note': 'per-round durations on stream 0 of rank 0 (every batch advanced by %d steps per round); median_value = nominal env-steps of a round / median' % C}

    # ---- the path's single collective: gather of episode statistics (terminal-class counts + env-steps of all finished
    # episodes of every rank) to rank 0 ----
    def episode_summary():
        tot = torch.zeros(5, dtype=torch.float64, device=dev)
        for env in envs:
            n = int(min(env._case_counter.item(), env.k_total))
            info = env.episodes.res_info[:n]; steps = env.episodes.res_steps[:n]
            fin = steps > 0
            for j, code in enumerate((_abi.INFO_REACHGOAL, _abi.INFO_COLLISION, _abi.INFO_TIMEOUT)):
                tot[j] += ((info == code) & fin).sum()
            tot[3] += steps[fin].sum(); tot[4] += fin.sum()
        return tot
    summ = episode_summary()
    if world > 1:
        gathered = [torch.empty_like(summ) for _ in range(world)]
        dist.all_gather(gathered, summ)
        summ = torch.stack(gathered).sum(dim=0)
    summ = summ.tolist()
    episodes = {'finished': int(summ[4]), 'success_rate': summ[0] / max(summ[4], 1), 'collision_rate': summ[1] / max(summ[4], 1),
                'timeout_rate': summ[2] / max(summ[4], 1), 'mean_steps': summ[3] / max(summ[4], 1),
                'note': 'all episodes finished so far on all ranks (gathered with one NCCL all_gather when n_gpus > 1); reference '
                        '500-case test suite: 0.43 / 0.57 / 0.006'}

    # ---- BASELINE config 2 taken literally: ONE batch of 4096 envs, nothing else on the GPU. (a) the same batch over and
    # over (its 2.6 MB of state stay in L2 -- and, inside a launch, in registers); (b) one batch in flight at a time but
    # rotating through all batches, so every launch reads its state from HBM. Auto-reset and scene refill included. ----
    def time_pair(g_step, g_fill, reps):
        """reps x (step graph on lane 0 || refill graph on side 0), CUDA events on lane 0 (the refills overlap the steps)."""
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sides[0].wait_stream(lanes[0])
        with torch.cuda.stream(lanes[0]):
            q0.record()
        for _ in range(reps):
            with torch.cuda.stream(lanes[0]):
                g_step.replay()
            with torch.cuda.stream(sides[0]):
                g_fill.replay()
        with torch.cuda.stream(lanes[0]):
            q1.record()
        barrier()
        tq = torch.tensor([q0.elapsed_time(q1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tq, op=dist.ReduceOp.MAX)
        return float(tq.item())
    n_ch = 4
    one = [envs[0]]
    g_same, f_same = stream_graph(0, [0], n_chunks=n_ch), stream_graph(0, [0], n_chunks=n_ch, step_fn=refill, side=True)   # one refill per step launch
    reps = max(3, int(0.03 / (n_ch * C * 8e-6)))
    time_pair(g_same, f_same, 2)
    b0 = env_steps_done(one)
    ms_same = time_pair(g_same, f_same, reps)
    done_same = env_steps_done(one) - b0
    g_rot, f_rot = stream_graph(0, list(range(pools))), stream_graph(0, list(range(pools)), step_fn=refill, side=True)
    time_pair(g_rot, f_rot, 1)
    b1 = env_steps_done()
    ms_rot = time_pair(g_rot, f_rot, 3)
    done_rot = env_steps_done() - b1
    single = {'value': world * done_same / (ms_same * 1e-3), 'unit': 'env-steps/s',
              'us_per_step': 1e3 * ms_same / (reps * n_ch * C),
              'rotating_value': world * done_rot / (ms_rot * 1e-3), 'rotating_us_per_step': 1e3 * ms_rot / (3 * pools * C),
              'note': 'config-literal: ONE %d-env batch in flight. value: the same batch stepped %d x %d steps back to back (state L2-resident between '
                      'launches); rotating_value: one batch in flight, rotating over %d batches (state from HBM). Both with auto-reset + scene refill '
                      '(side stream); env-steps counted by the kernel' % (B, reps * n_ch, C, pools)}
    del g_same, g_rot, f_same, f_rot

    # ---- roofline of the dominant kernel (the step kernel of the timed region: crowdsim_step_n with C steps per launch): a
    # single-stream graph of one launch per batch, no bookkeeping / resets in between, replayed R times; CUDA events on the
    # launching stream; per-launch duration = elapsed / (R * pools). The batches rotate: each launch reads its state from HBM.
    # Algorithmic bytes per launch = C steps x B envs x 634 B (SURVEY.md 8d: the per-env-step figure x the env-steps a launch
    # performs); the launch's actual DRAM traffic is lower -- that is the point of keeping the state in registers. ----
    def kernel_us(n):
        """Average duration of one step launch (n env-steps) in the bench's own steady state: episode bookkeeping and
        auto-reset ON (finished envs install their next scene and go on -- without resets every episode would run out into
        a quiet scene, the cheapest input there is), the scene refills run between the timed replays, untimed."""
        g_fill = stream_graph(0, list(range(pools)), step_fn=refill)
        g_k = stream_graph(0, list(range(pools)), step_fn=(lambda e: e.step_n(n)) if n > 1 else (lambda e: e.step()))
        tot = 0.0
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(R + 1):
            with torch.cuda.stream(lanes[0]):
                g_fill.replay()
                q0.record(); g_k.replay(); q1.record()
            torch.cuda.synchronize()
            if r > 0:
                tot += q0.elapsed_time(q1)
        return tot / (R * pools)
    peak, peak_src = load_peaks()
    R = max(3, min(20, 1200 // pools))
    CR = C if N <= 5 else 1                                  # env-steps of ONE kernel launch (N > 5: crowdsim_step_n = n launches of the crowd kernel)
    k_avg = kernel_us(CR)
    k1_avg = kernel_us(1) if CR > 1 else k_avg
    achieved = CR * B * bytes_per_env / (k_avg * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'step_traffic.json')
    if os.path.exists(tpath) and N == 5 and B == 4096:
        tj = json.load(open(tpath))
        if tj.get('steps_per_launch', 1) == CR:
            traffic = tj['dram_bytes_read'] + tj['dram_bytes_write']      # from the committed ncu --set full capture, per launch
    roofline = {'bound': 'hbm', 'kernel': ('cs::step_flat_kernel<%d, MULTI> (crowdsim_step_n, %d env-steps per launch)' % (N, CR)) if N <= 5 and CR > 1 else ('cs::step_flat_kernel' if N <= 5 else 'cs::step_kernel<MID> (crowd kernel, step_mid.cuh)'),
                'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                'algorithmic_bytes_per_launch': CR * B * bytes_per_env, 'avg_launch_us': 1e3 * k_avg, 'env_steps_per_launch': CR * B,
                'how': 'CUDA events around each of %d replays of a single-stream graph of %d back-to-back step launches (one per rotating batch, bookkeeping + auto-reset on, scene refills between the replays untimed)' % (R, pools),
                'single_step_kernel': {'avg_launch_us': 1e3 * k1_avg, 'achieved': B * bytes_per_env / (k1_avg * 1e-3) / 1e9,
                                       'frac': B * bytes_per_env / (k1_avg * 1e-3) / 1e9 / peak, 'note': 'crowdsim_step (one env-step per launch), same measurement (steady-state scenes, bookkeeping + auto-reset on); round 1 reported 0.039 from launches that ran past the ends of their episodes (no resets: quieter scenes)'},
                'timed_region_GBps': (live_total / world) * bytes_per_env / (ms_max * 1e-3) / 1e9,
                'timed_region_frac': (live_total / world) * bytes_per_env / (ms_max * 1e-3) / 1e9 / peak,
                'timed_region_note': 'algorithmic bytes of all steps of the timed region / its duration, with %d independent batches in flight' % S}

    # ---- supplementary: the single-step kernel when the batch fills the chip (1 Mi envs in ONE launch, state = 665 MB) ----
    scale = None
    if rank == 0 and not args.no_scale:
        Bs = 1 << 20
        big = BatchedCrowdSim(Bs, device=dev)
        big.configure(default_config(human_num=N, test_sim=args.rule, train_val_sim=args.rule))
        big.set_robot_policy('orca')
        big.reset_seeds(torch.arange(Bs, dtype=torch.int64) % (2 ** 31) + 5000, rule=args.rule)
        with torch.cuda.stream(main):
            for _ in range(12):
                big.step()                                   # into the episodes (agents meet around step 12-20)
            gb = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gb, stream=main):
            for _ in range(8):
                big.step()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(main):
            s0.record(); gb.replay(); s1.record()
        torch.cuda.synchronize()
        us = s0.elapsed_time(s1) / 8 * 1e3
        scale = {'envs_per_launch': Bs, 'us_per_launch': us, 'env_steps_per_s': Bs / us * 1e6, 'achieved_GBps': Bs * bytes_per_env / us / 1e3,
                 'roofline_frac': Bs * bytes_per_env / us / 1e3 / peak, 'note': 'single-step kernel only, no resets; shows the issue-bound regime when the chip is full'}
        del big, gb

    # ---- e2e: the public host-facing API (HostStepper): pinned HOST buffers in and out every step. The robot is
    # driven from the host like the reference's Explorer loop does it: action up, obs/reward/done/info (+ the robot's
    # next ORCA decision) down, host waits for the results before the next step. ----
    import numpy as np
    from crowdnav_b200.batched import HostStepper
    P = max(1, min(pools, args.e2e_batches))
    steppers = []
    for env in envs[:P]:
        env.reset_seeds(rule=args.rule, use_queue=True)      # fresh scenes (the step-only pass ran past terminal states)
        env.set_robot_policy('external_xy')
        e2e_transfer = args.e2e_transfer if args.e2e_transfer != 'auto' else ('direct' if B * (16 * N + 34) < (1 << 20) else 'copy')
        steppers.append(HostStepper(env, next_orca_action=True, obs=args.e2e_obs, transfer=e2e_transfer if args.e2e_obs == 'f32' else 'copy'))
    for st in steppers:
        st.step()
        for _ in range(40):                                  # into the episodes
            st.h_action.copy_(st.h_next_action); st.step()
    ke = 400

    def e2e_rate(group, n):
        """Round-robin over the batches in `group`; each visit = wait for the batch's previous step (results in host
        memory), host-side "policy" (apply the decision the device computed), enqueue its next step."""
        for st in group:
            st.launch()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            for st in group:
                st.wait()
                np.copyto(st.np_action, st.np_next_action)
                st.launch()
        for st in group:
            st.wait()
        dt_ = time.perf_counter() - t0
        t = torch.tensor([dt_], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * B * n * len(group) / float(t.item())

    from crowdnav_b200.batched import HostStepperGroup
    group = HostStepperGroup(steppers)

    def e2e_native(n):
        """The same round-robin with the loop in native code (HostStepperGroup.run = crowdsim_host_pump): wait, hand the
        device's decision back as the next action (host memcpy), launch -- per batch-step, for every batch."""
        group.start()
        barrier()
        t0 = time.perf_counter()
        group.run(n)
        group.wait()
        dt_ = time.perf_counter() - t0
        t = torch.tensor([dt_], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * B * n * len(steppers) / float(t.item())

    e2e_single = e2e_rate(steppers[:1], ke)                  # one batch, host blocks on every step (the reference's loop shape)
    e2e_python = sorted(e2e_rate(steppers, ke) for _ in range(3))[1] if P > 1 else e2e_single  # P batches in flight, Python round-robin, median of 3
    e2e_value = sorted(e2e_native(2 * ke) for _ in range(3))[1]                                # the same, round-robin in native code
    stepper = steppers[0]
    h2d, d2h = stepper.h2d_bytes, stepper.d2h_bytes
    launches_note = 'timed region: %d rounds x (%d crowdsim_step_n launches of %d env-steps + %d scene-prefetch launches); per round every stream replays its graph of step launches and every side stream its graph of refills' % (rounds, pools, C, pools)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, sample = cpu_oracle_rate(args)
        cpu = {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
               'sample': sample + '; C restatement of the reference loop (oracle/crowdsim_oracle.c), OpenMP over envs'}

    # ---- second half of the metric ("500-case success/collision parity"): BASELINE config 1's 500 test cases (seeds 1000..1499,
    # ORCA robot) through BatchedExplorer on this GPU, against the reference's recorded outcome (tests/golden, SURVEY App. B).
    # Outside every timed region; a failure here is reported, it does not take the throughput line down.
    parity = None
    if rank == 0:
        try:
            from crowdnav_b200.explorer import BatchedExplorer
            penv = BatchedCrowdSim(512, device=dev)
            penv.configure(default_config(human_num=5))
            st500 = BatchedExplorer(penv, 'orca', gamma=0.9).run_k_episodes(500, 'test')
            ref500 = {'success': 213, 'collision': 284, 'timeout': 3, 'timeout_cases': [118, 168, 224], 'env_steps': 15190}
            got500 = {k_: st500[k_] for k_ in ref500}
            parity = {'cases': 500, 'ours': got500, 'reference': ref500, 'match': got500 == ref500,
                      'note': 'test.py --policy orca flow (5 humans, circle_crossing, invisible robot); per-case bit-exact parity is in tests/'}
        except Exception as ex:                              # noqa: BLE001
            parity = {'error': repr(ex)}

    if rank == 0:
        line = {'metric': METRIC, 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': K, 'warmup': W,
                'ms_per_step': ms_max / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f64 state + f32 ORCA solver', 'data': 'synthetic',
                'config': {'workload': WORKLOAD % (B, N, args.rule),
                           'envs_per_gpu': B, 'humans': N, 'l2': 'inputs larger than L2: %d rotating independent batches = %.0f MB of state' % (pools, pools * B * bytes_per_env / 1e6),
                           'batches_in_flight': S, 'steps_per_launch': C,
                           'parallelism': 'independent envs sharded over %d GPU(s), no data-path collective' % world},
                'value_is': '%d independent %d-env batches in flight on %d streams (weak scaling unit = one GPU with its %d batches); the config-literal one-batch number is `single_batch`' % (S, B, S, pools),
                'timed_region': {'timed_steps': K, 'envs_per_step': pools * B, 'env_steps_per_env_per_step': C, 'ms': ms_max,
                                 'warmup_steps_done': warm_rounds,
                                 'note': 'K steps (one crowdsim_step_n launch per batch each) run back to back without a gap (streams joined only at the two ends of the region); ms_per_step = ms / K; '
                                         'every env was advanced %d env-steps before the region (steady mix of episode phases)' % (warm_rounds * C)},
                'rounds': round_stats,
                'env_steps': {'performed': live_total, 'nominal': world * pools * B * C * K,
                              'note': 'value = performed / time; performed is counted by the step kernel (episode step counters), nominal = envs x steps; they differ only if envs waited for a scene refill'},
                'clocks': clocks, 'gpu_launches': int(launches), 'gpu_launches_note': launches_note,
                'e2e': {'value': e2e_value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                        'steps': 2 * ke, 'batches_in_flight': P, 'transfer': steppers[0].transfer, 'single_batch_blocking': e2e_single, 'python_round_robin': e2e_python, 'observation': args.e2e_obs,
                        'note': 'HostStepperGroup.run() (round-robin in native code: crowdsim_host_pump; python_round_robin = the same loop written in Python with HostStepper.launch()/wait()) over %d independent %d-env batches: per batch-step a pinned host action buffer goes up and obs (%s)/reward/dmin/done/info/next ORCA action come down (byte counts are per batch-step), the host waits for a batch\'s results before it feeds that batch again; single_batch_blocking = one batch, host blocks on every step' % (P, B, 'float32 px,py,vx,vy per human' if args.e2e_obs == 'f32' else 'float64 state arrays')},
                'single_batch': single, 'parity_500_cases': parity, 'episodes': episodes, 'roofline': roofline, 'scale': scale, 'cpu_baseline': cpu}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
