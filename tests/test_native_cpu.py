"""CPU fuzz of the CUDA solver's arithmetic: orca_device.cuh / orca_spec.cuh are __host__ __device__, so the exact code the
kernels run is compiled for the host (nvcc, --fmad=false, -ffp-contract=off) and compared bit for bit with the C oracle on
millions of random ORCA problems -- line construction (at several time horizons and time steps), sequential lp2/lp3, the speculative lp1_all + lp2_scan path and the
lane-parallel formulation of lp3 (independent per-line sub-problems + outer scan). See tests/native/lp_fuzz.cu."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def fuzz_binary(tmp_path_factory):
    from crowdnav_b200 import build
    exe = str(tmp_path_factory.mktemp('native') / 'lp_fuzz')
    cmd = [build._nvcc(), '-O2', '--fmad=false', '-Xcompiler', '-ffp-contract=off', '-std=c++17', '-gencode',
           'arch=compute_100a,code=sm_100a', '-diag-suppress', '20013', '-o', exe, os.path.join(ROOT, 'tests', 'native', 'lp_fuzz.cu')]
    subprocess.check_call(cmd)
    return exe


@pytest.mark.parametrize('seed', [1, 2, 3])
def test_host_compiled_solver_matches_oracle_bitwise(fuzz_binary, seed):
    out = subprocess.run([fuzz_binary, '1000000', str(seed)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-500:]
    fields = dict(kv.split('=') for kv in out.stdout.strip().split()[1:])
    assert int(fields['cases']) == 1000000
    # the interesting branches are really exercised
    assert int(fields['lp3_needed']) > 100000 and int(fields['speculative_checked']) > 500000
    assert int(fields['overlapping_pairs']) > 100000 and int(fields['forced_parallel_lines']) > 100000
    assert int(fields['sorted_lists']) == 1000000                                                    # part H
    assert int(fields['lane_lp3_checked']) == int(fields['lp3_needed'])                              # part F
    assert int(fields['neighbour_orders']) == 4000000 and int(fields['neighbour_ties']) > 1000000    # part E, M = 5, 4, 2, 1
    # line construction away from the default 5 s horizon / 0.25 s step (3 of 4 cases each)
    assert int(fields['other_horizon']) > 700000 and int(fields['other_time_step']) > 700000
