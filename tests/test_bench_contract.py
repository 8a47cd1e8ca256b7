"""bench.py's reference arm runs here (no GPU): one JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '1', '--model', 'rc', '--num', '64'], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step',
              'higher_is_better', 'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in line, k
    assert line['impl'] == 'reference' and line['value'] > 0 and line['unit'] == 'rays/s'
    assert line['e2e'] == {'value': line['value'], 'unit': 'rays/s', 'h2d_bytes_per_step': 0,
                           'd2h_bytes_per_step': 0}
    cb = line['cpu_baseline']
    assert cb['kind'] in ('reference', 'port') and cb['cores'] >= 1 and 'sample' in cb
    if cb['kind'] == 'reference':               # baseline/_ref installed: the unmodified Python reference
        assert cb['port']['kind'] == 'port' and cb['port']['value'] > cb['value']
        assert 'trace_grid' in cb['sample']
    assert 'workload' in line['config'] and 'model' not in line['config']


def test_other_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2'],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ''


def test_b200_arm_line_on_the_dry_run_engine():
    """The B200 arm's host code end to end (tests/dry_bench.py: CUDA entry points replaced by the
    oracle-backed stand-in): the JSON line carries every key of the bench contract, both step
    submission modes."""
    for extra, mode in ((['--no-graph'], 'eager launches'), ([], 'one CUDA graph replay per step')):
        p = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'dry_bench.py'), '--steps', '2', '--warmup',
                            '1', '--num', '24'] + extra, capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-3000:]
        line = json.loads(p.stdout.strip().splitlines()[-1])
        for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
                  'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches',
                  'roofline', 'cpu_baseline'):
            assert k in line, k
        assert line['steps'] == 2 and line['warmup'] >= 3 and line['n_gpus'] == 1 and line['dtype'] == 'f64'
        assert line['scaling'] == 'weak' and line['vs_baseline'] is None and line['higher_is_better'] is True
        assert 'workload' in line['config'] and 'model' not in line['config']
        assert set(line['e2e']) >= {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'}
        assert line['e2e']['h2d_bytes_per_step'] > 0 and line['e2e']['d2h_bytes_per_step'] >= 16*3604
        roof = line['roofline']
        for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
            assert k in roof, k
        assert roof['bound'] == 'fp64' and roof['unit'] == 'TFLOP/s' and roof['hbm']['unit'] == 'GB/s'
        assert abs(roof['frac'] - roof['achieved']/roof['peak']) < 1e-12
        cb = line['cpu_baseline']
        for k in ('value', 'unit', 'cores', 'kind', 'sample'):
            assert k in cb, k
        assert set(line['clocks']) >= {'sm_mhz', 'sm_max_mhz', 'reasons'}
        assert line['step_submission'].startswith(mode)
        assert line['parity_vs_reference']['bit_identical_p_d_op'] is True


def test_b200_arm_dumps_the_last_step_on_the_dry_run_engine(tmp_path):
    """--dump-outputs DIR: the last timed step's records as float64 .npy files, the same from
    run to run with the same arguments."""
    import numpy as np
    runs = []
    for k in range(2):
        out = tmp_path / str(k)
        p = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'dry_bench.py'), '--steps', '2', '--warmup',
                            '1', '--num', '24', '--no-e2e', '--no-cpu-baseline', '--dump-outputs', str(out)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-3000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])['steps'] == 2
        runs.append({f.name: np.load(f) for f in sorted(out.iterdir())})
    a, b = runs
    assert set(a) == {'ray_index.npy', 'p.npy', 'd.npy', 'op.npy', 'abr.npy', 'status.npy', 'fail_surf.npy',
                      'spot_sums.npy'}
    n = 3*3*24*24
    assert a['p.npy'].shape == (3, n) and a['abr.npy'].shape == (2, n) and a['status.npy'].shape == (n,)
    assert np.array_equal(a['ray_index.npy'], np.arange(n))
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k], equal_nan=True), k
    assert 0 < (a['status.npy'] == 0).sum() < n


def test_b200_arm_two_ranks_on_the_dry_run_engine():
    """world size 2 over gloo (dry-run engine): the eager multi-rank step loop with its asynchronous
    all-gather + combine, max-over-ranks timing and the shard mode's equal-work ranges produce
    ONE line, from rank 0, with whole-job ray counts."""
    import socket
    for mode, rays, scaling in (('replica', 2*5184, 'weak'), ('shard', 5184, 'strong')):
        with socket.socket() as s:
            s.bind(('127.0.0.1', 0))
            port = s.getsockname()[1]
        procs = []
        for r in range(2):
            env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE='2', MASTER_ADDR='127.0.0.1',
                       MASTER_PORT=str(port))
            procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, 'tests', 'dry_bench.py'), '--gpus', '2',
                                           '--steps', '3', '--warmup', '1', '--num', '24', '--mode', mode],
                                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, env=env))
        outs = [p.communicate(timeout=600) for p in procs]
        assert all(p.returncode == 0 for p in procs), outs[0][1][-2000:] + outs[1][1][-2000:]
        assert outs[1][0].strip() == ''
        line = json.loads(outs[0][0].strip().splitlines()[-1])
        assert line['n_gpus'] == 2 and line['scaling'] == scaling and line['steps'] == 3
        assert line['config']['rays_per_step'] == rays and line['step_submission'] == 'eager launches'
        assert line['rank_imbalance']['kernel_ms_max_over_ranks'] >= line['rank_imbalance']['kernel_ms_min_over_ranks']
        assert (line['rank_imbalance']['shard_balance'] is not None) == (mode == 'shard')
        assert line['e2e']['value'] > 0 and 'cpu_baseline' not in line
        c = line['collectives']            # 3 steps, default --gather-every 8: one all-gather for all of them
        assert c == {'all_gathers_in_timed_region': 1, 'steps_per_all_gather': 3,
                     'payload_bytes_per_rank_per_gather': 3*9*16*8, 'last_combined_ok': True}


def test_default_engine_paths_of_the_new_host_functions():
    """tests/dry_api.py: one-launch bisection, batched set_vig, post-import update, 'aim pt' pupils, the
    two-stage analyses, astigmatism / Coddington, real image heights (reverse path through the drop-in
    trace_raw), wide-angle aiming, set_pupil -- each through its default (engine) code path on the
    dry-run stand-in."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'dry_api.py')], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    assert 'ALL DEFAULT-ENGINE PATHS OK' in p.stdout
