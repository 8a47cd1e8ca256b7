#!/usr/bin/env python3
"""bench.py -- rays/sec (fp64) through a sequential model on B200(s).

Metric (BASELINE.json): rays/sec in fp64 through an N-surface sequential model.
Default workload: BASELINE configs[1] -- double Gauss (13 interfaces), 3 fields x 3
wavelengths x 512 x 512 pupil grid = 2,359,296 rays per step, apertures checked,
start rays generated on the device, per-ray last-segment records (p, d, op,
status, fail_surf: 64 B) + transverse aberration (16 B) written to HBM,
per-(field, wvl) spot sums reduced.  A step = one pass over that grid.
`--model rc|evenasph|cellphone|zoom52` selects the other BASELINE configurations
(their pupil sampling is the default `--num`).

Multi-GPU (`--gpus N` under torchrun):
  --mode replica (default)  weak scaling: every rank traces a full replica of the grid
                            on its own GPU; value = N x rays / max-rank time
  --mode shard              strong scaling: the grid's chunk space (field-major, then
                            wavelength, then pupil rows) is cut into N contiguous ranges,
                            one per rank (parallel.shard_chunks); value = rays / max-rank time
In both the only collective is the all-gather of the [n_tiles, 16] spot sums; the sums of
`--gather-every` K consecutive steps (default 8) travel in ONE asynchronous
all_gather_into_tensor (NCCL's stream) and are combined by one rt_combine_summaries launch, so
every step's combined sums exist before the timed region ends at 1/K of the collective count.

  python bench.py --gpus N --steps K --warmup W            (this repo's engine)
  python bench.py --impl reference --gpus N --steps K ...  (CPU arm: the UNMODIFIED Python
        reference from baseline/_ref on all host cores -- its own trace.trace_grid ->
        trace_raw, baseline/reference_arm.py -- on a bounded sample of the same workload;
        the C port oracle/rt_oracle.c is timed next to it.  Falls back to the port alone
        if baseline/_ref is not installed.)

One JSON line on stdout (rank 0).  DESIGN.md "Measurement" says how every field
is obtained.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'rays/sec (fp64) through N-surface seq model'
UNIT = 'rays/s'


# BASELINE.json configs -> fixture model and pupil samples per side
WORKLOADS = {
    'singlet': (7, 'BASELINE configs[0]'),
    'dblgauss': (512, 'BASELINE configs[1]'),
    'rc': (1024, 'BASELINE configs[2]'),
    'evenasph': (256, 'BASELINE configs[3], Zemax EVENASPH import'),
    'cellphone': (256, 'BASELINE configs[3] geometry on the cell-phone lens (8 RadialPolynomial surfaces)'),
    'zoom52': (1024, 'BASELINE configs[4]'),
}

# --dump-outputs: rays sampled from the last timed step (9 float64 records + status + fail_surf
# = 88 B a ray, 23 MB at 2^18 rays)
DUMP_MAX_RAYS = 1 << 18
DUMP_SEED = 20261017


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--model', default='dblgauss', choices=sorted(WORKLOADS))
    ap.add_argument('--num', type=int, default=None, help='pupil samples per side (default: the BASELINE config)')
    ap.add_argument('--mode', default='replica', choices=['replica', 'shard'])
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='eager step loop instead of CUDA graph replay')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--gather-every', type=int, default=8,
                    help='multi-GPU: steps whose spot sums share one all-gather (1 = a collective per step)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the results of the last timed step to DIR/<name>.npy (rank 0; a fixed '
                         'seeded sample of at most %d rays, float64)' % DUMP_MAX_RAYS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.baseline_num = WORKLOADS[args.model][0]
    if args.num is None:
        args.num = args.baseline_num
    return args


def load_model(name):
    from rayoptics_b200 import model as M
    return M.OpticalModel.load(os.path.join(ROOT, 'tests', 'golden', 'models', name + '.json'))


# ---------------------------------------------------------------- flop model
# Algorithmic work per ray per interface, from the reference's algebra
# (SURVEY.md 8(d) table; add/mul/sub = 1, fma = 2, div = 1, sqrt = 1).
def interface_flops(desc, n_wild_newton=3.3):
    tfrm = 3 if desc.has_tfrm == 0 else 33
    closest = 12
    k = desc.n_coefs
    if desc.profile == 0:
        isect, nrm = 28, 13
    elif desc.profile == 1:
        isect, nrm = 41, 15
    else:
        isect, nrm = n_wild_newton*(46 + 5*k), 20 + 3*k
    act = {0: 33, 1: 18}.get(desc.mode, 0)
    return dict(tfrm=tfrm, closest=closest, isect=isect, dst=3, nrm=nrm, ap=4, act=act)


def flops_by_outcome(descs):
    """cum[k] = flops of a ray that completes interface k; plus partial costs."""
    n = len(descs)
    start = 20 + 6                      # start-ray generation + transverse aberration
    obj = interface_flops(descs[0])
    cum = [start + obj['isect'] + obj['nrm']]
    parts = [None]
    for k in range(1, n):
        f = interface_flops(descs[k])
        f['tfrm'] = interface_flops(descs[k - 1])['tfrm']
        parts.append(f)
        cum.append(cum[-1] + sum(f.values()))
    return cum, parts


def algorithmic_flops(descs, status, fail_surf):
    cum, parts = flops_by_outcome(descs)
    cum = np.array(cum, dtype=np.float64)
    n_ifc = len(descs)
    total = float((status == 0).sum())*cum[-1]
    for st in (1, 2, 3, 5):
        m = status == st
        if not m.any():
            continue
        ks = np.bincount(fail_surf[m], minlength=n_ifc)
        for k, cnt in enumerate(ks):
            if cnt == 0 or k == 0:
                continue
            f = parts[k]
            if st in (1, 5):
                w = cum[k - 1] + f['tfrm'] + f['closest'] + f['isect']
            elif st == 3:
                w = cum[k] - f['act']
            else:
                w = cum[k]
            total += cnt*w
    return total, cum[-1]


# ------------------------------------------------------------ clock sampling
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                       '-lms', '100', '-i', str(gpu_index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, reasons, pw = [], [], set(), []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(',')]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); smax.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                                'sw_power_cap'), c[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)),
                       reasons=sorted(reasons), samples=len(sm), power_w_max=float(max(pw)))
        return out


# ------------------------------------------------------------- CPU baseline
def host_grid_spec(opm, num):
    """Host-only grid spec with chief-ray reference image points from the oracle."""
    from oracle import rt_oracle
    from rayoptics_b200 import _abi, table as T, engine as E
    sm = opm.seq_model
    descs, n_by_wvl, _ = T.describe_model(sm)
    fields = opm.optical_spec.fov.fields
    g0 = E.grid_spec_for_model(opm, 1, wvls=[sm.central_wavelength()], pupil_range=(0.0, 0.0),
                               apply_vignetting=False)
    o0 = _abi.make_opts(first_surf=1, last_surf=len(descs) - 2, check_apertures=False)
    r0 = rt_oracle.trace_grid(g0.c_spec(), descs, n_by_wvl, 0, g0.n_rays, o0)
    ref = r0['last'][0:2].T.copy()
    ref_fw = np.repeat(ref[:, None, :], len(sm.wvlns), axis=1)
    spec = E.grid_spec_for_model(opm, num, ref_img=ref_fw)
    return spec, descs, n_by_wvl


def cpu_trace(spec, descs, n_by_wvl, r0, r1, threads):
    from oracle import rt_oracle
    from rayoptics_b200 import _abi
    opts = _abi.make_opts(first_surf=1, last_surf=len(descs) - 2, check_apertures=True)
    t0 = time.perf_counter()
    r = rt_oracle.trace_grid(spec.c_spec(), descs, n_by_wvl, r0, r1, opts, n_threads=threads,
                             want_last=False)
    return time.perf_counter() - t0, r


def port_arm(spec, descs, n_by_wvl, r0, r1, target_s=6.0, scaling=True):
    """oracle/rt_oracle.c (the C port of trace_raw + start rays + transverse aberration) on a
    persistent pthread pool with dynamic scheduling, output buffers allocated and first touched
    before the timed calls; only the C call is timed.  Thread scaling at 1 / 32 / all."""
    from oracle import rt_oracle
    from rayoptics_b200 import _abi
    cores = os.cpu_count() or 1
    opts = _abi.make_opts(first_surf=1, last_surf=len(descs) - 2, check_apertures=True)
    out = {'unit': UNIT, 'kind': 'port', 'cores': cores, 'threads_scaling': {}}
    runner = None
    for th in (sorted({1, min(8, cores), min(16, cores), min(32, cores), min(64, cores), cores})
               if scaling else [cores]):
        runner = rt_oracle.GridRunner(spec, descs, n_by_wvl, opts, r1 - r0, th)
        n_w = r1 - r0 if th > 1 else min(r1 - r0, 50000)
        runner.run(r0, r0 + n_w)                                        # warm-up, first touch
        reps, tot, budget = 0, 0.0, (target_s if th == cores else target_s/6)
        while tot < budget and reps < 200:
            tot += runner.run(r0, r0 + n_w)
            reps += 1
        out['threads_scaling'][str(th)] = n_w*reps/tot
        if th == cores:
            out['value'] = n_w*reps/tot
            out['parallel_speedup'] = out['value']/out['threads_scaling']['1']
            out['sample'] = (f'{reps} x {n_w} rays of the same grid, oracle/rt_oracle.c on a persistent pool of '
                             f'{cores} pthreads (dynamic blocks of 2048 rays), buffers pre-touched, C call only')
    return out, runner


def python_reference_arm(model, steps, warmup, step_s=1.5):
    """The unmodified Python reference (baseline/_ref) on one worker process per host core, run
    by baseline/reference_arm.py in a fresh interpreter (no CUDA context, no NCCL in the
    workers' parent).  Returns the arm's dict, or (None, reason)."""
    cmd = [sys.executable, os.path.join(ROOT, 'baseline', 'reference_arm.py'), '--model', model,
           '--steps', str(steps), '--warmup', str(warmup), '--step-s', str(step_s)]
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=ROOT)
        out = json.loads(p.stdout.strip().splitlines()[-1])
    except Exception as e:      # noqa: BLE001
        return None, repr(e)
    if 'unavailable' in out:
        return None, out['unavailable']
    return out, None


def parity_vs_oracle(spec, descs, n_by_wvl, r0, r1, cores, gpu):
    """SURVEY 8(d): ray-intercept RMS / max-abs at the image interface between the
    engine's records of the timed steps and the oracle on the same grid rays, plus
    exact equality of status / fail_surf.  `gpu(r0, r1)` returns host copies."""
    from oracle import rt_oracle
    from rayoptics_b200 import _abi
    opts = _abi.make_opts(first_surf=1, last_surf=len(descs) - 2, check_apertures=True)
    ref = rt_oracle.trace_grid(spec.c_spec(), descs, n_by_wvl, r0, r1, opts, n_threads=cores)
    g = gpu(r0, r1)
    ok = ref['status'] == 0
    dxy = g['p'][0:2][:, ok] - ref['last'][0:2][:, ok]
    dist = np.sqrt((dxy**2).sum(0))
    bit_equal = all(np.array_equal(a, b, equal_nan=True) for a, b in (
        (g['p'], ref['last'][0:3]), (g['d'], ref['last'][3:6]), (g['op'], ref['op']),
        (g['abr'], ref['abr'])))
    return {'rays': int(r1 - r0), 'rays_ok': int(ok.sum()),
            'intercept_rms_mm': float(np.sqrt((dist**2).mean())) if ok.any() else 0.0,
            'intercept_max_abs_mm': float(dist.max()) if ok.any() else 0.0,
            'status_equal': bool(np.array_equal(g['status'], ref['status'])),
            'fail_surf_equal': bool(np.array_equal(g['fail_surf'], ref['fail_surf'])),
            'bit_identical_p_d_op_abr': bool(bit_equal), 'target_mm': 1e-10,
            'against': 'oracle/rt_oracle.c (pinned on the reference golden vectors), '
                       'tile field 1 / wvl 1 of the timed grid'}


def parity_vs_reference_golden(model, opm, tab):
    """Engine vs tests/golden/vectors/<model>_grid.npz: the model's fields x wavelengths at a
    reduced pupil grid traced by the body of the reference's own trace_grid loop in the build
    container (tests/golden/make_golden_grids.py).  Outside every timed region."""
    import torch
    from rayoptics_b200 import engine as E
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'vectors', model + '_grid.npz'))
    grid = E.grid_for_model(opm, tab, int(z['num']))
    r = E.trace_grid(tab, grid)
    torch.cuda.synchronize()
    status = r.status.cpu().numpy()
    ok = z['status'] == 0
    p = r.p.cpu().numpy().T
    dxy = p[ok, 0:2] - z['p'][ok, 0:2]
    dist = np.sqrt((dxy**2).sum(1))
    bit = (np.array_equal(p[ok], z['p'][ok]) and np.array_equal(r.d.cpu().numpy().T[ok], z['d'][ok])
           and np.array_equal(r.op.cpu().numpy()[ok], z['op'][ok]))
    grid.close()
    return {'rays': int(ok.size), 'rays_ok': int(ok.sum()), 'pupil_grid': int(z['num']),
            'intercept_rms_mm': float(np.sqrt((dist**2).mean())),
            'intercept_max_abs_mm': float(dist.max()),
            'status_equal': bool(np.array_equal(status, z['status'])),
            'bit_identical_p_d_op': bool(bit), 'target_mm': 1e-10,
            'against': 'rayoptics.raytr.trace.trace_safe/trace_base/raytrace.trace_raw of the '
                       'reference (golden vectors generated in the build container)'}


def cpu_baseline(args, opm, gpu=None):
    """CPU side of the main line (rank 0, N=1): the Python reference on all cores on a bounded
    sample (kind "reference") when baseline/_ref is installed, and the C port next to it."""
    num = args.num
    spec, descs, n_by_wvl = host_grid_spec(opm, num)
    per_tile = num*num
    tile = min(4, spec.n_tiles - 1)
    r0 = tile*per_tile
    r1 = r0 + min(per_tile, 1 << 20)
    port, _ = port_arm(spec, descs, n_by_wvl, r0, r1)
    ref, why = None, None
    try:
        ref, why = python_reference_arm(args.model, steps=6, warmup=1)
    except Exception as e:      # noqa: BLE001 - never lose the bench line over the baseline
        why = repr(e)
    if ref is not None:
        out = dict(ref, port=port)
    else:
        out = dict(port, reference_unavailable=str(why))
    if gpu is not None:
        try:
            out['parity'] = parity_vs_oracle(spec, descs, n_by_wvl, r0, r1, port['cores'], gpu)
        except Exception as e:      # noqa: BLE001 - never lose the bench line over the checker
            out['parity'] = {'error': repr(e)}
    return out


# ------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    opm = load_model(args.model)
    spec, descs, n_by_wvl = host_grid_spec(opm, args.num)
    n = spec.n_rays
    port, runner = port_arm(spec, descs, n_by_wvl, 0, min(n, 1 << 22), target_s=4.0)
    ref, why = python_reference_arm(args.model, args.steps, args.warmup)
    if ref is not None:
        val, ms = ref['value'], ref['ms_per_step']
        base = dict(ref, port=port)
    else:       # baseline/_ref missing: the port is the arm, K steps over (a bounded part of) the grid
        n_s = min(n, 1 << 22)
        for _ in range(max(args.warmup, 1)):
            runner.run(0, n_s)
        t_tot = sum(runner.run(0, n_s) for _ in range(args.steps))
        val, ms = n_s*args.steps/t_tot, 1e3*t_tot/args.steps
        base = dict(port, value=val, reference_unavailable=str(why),
                    sample=f'{args.steps} steps x {n_s} rays, ' + port['sample'].split(', ', 1)[1])
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT,
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms, 'higher_is_better': True,
            'scaling': 'weak' if args.mode == 'replica' else 'strong',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config_dict(args, opm, spec, args.gpus),
            'cpu_baseline': base,
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def config_dict(args, opm, grid, world):
    sm = opm.seq_model
    tag = WORKLOADS[args.model][1] if args.num == args.baseline_num else 'reduced pupil sampling'
    n_rays = grid.n_rays
    mode = (f'replica-per-gpu x{world} (weak scaling)' if args.mode == 'replica' else
            f'grid chunk space sharded over {world} gpu(s) (strong scaling)')
    return {'workload': f'{args.model}: {sm.get_num_surfaces()} interfaces, {grid.n_fields} fields x '
                        f'{grid.n_wvls} wvls x {args.num}x{args.num} pupil ({tag})',
            'rays_per_step_per_gpu': n_rays if args.mode == 'replica' else -(-n_rays//world),
            'rays_per_step': n_rays*world if args.mode == 'replica' else n_rays,
            'check_apertures': True,
            'output': 'last segment p,d + op + status + fail_surf (64 B/ray) + transverse '
                      'aberration (16 B/ray) + per-(field,wvl) spot sums',
            'parallelism': mode + (f', the [n_tiles,16] spot sums of every {max(1, min(args.gather_every, args.steps))} steps '
                                   'all-gathered together' if world > 1 else ''),
            'l2': 'no HBM input is re-read (start rays are generated on-chip); each step writes '
                  f'{n_rays*80/1e6:.0f} MB of results per grid (L2: 126 MB)'}


def dump_outputs(out_dir, res, first_ray):
    """Write what the timed step returned to its caller -- the per-ray records of ``res`` and
    the per-(field, wvl) spot sums -- as float64 .npy files under ``out_dir``.  Grids of more
    than DUMP_MAX_RAYS rays are sampled at ray indices drawn once from a fixed seed, so two
    builds run with the same arguments write comparable files; ``ray_index.npy`` holds the
    sampled rays' indices in the whole grid."""
    os.makedirs(out_dir, exist_ok=True)
    n = res.n
    if n > DUMP_MAX_RAYS:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MAX_RAYS, replace=False))
    else:
        idx = np.arange(n)
    arrays = {'ray_index': first_ray + idx}
    for k in ('p', 'd', 'op', 'abr', 'status', 'fail_surf'):
        arrays[k] = getattr(res, k).cpu().numpy()[..., idx]
    arrays['spot_sums'] = res.summary.cpu().numpy()
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), np.ascontiguousarray(a, dtype=np.float64))


# ----------------------------------------------------------------- B200 arm
def kernel_name(tab_descs, lean_ok=True):
    poly = any(d.profile > 1 for d in tab_descs)
    general = any(d.has_tfrm != 0 or d.n_apertures != 0 or d.phase_kind != 0 or d.profile == 6
                  for d in tab_descs)
    if general:
        return 'k_trace_grid<0,1,1,0>'
    return 'k_trace_grid_lean<0,1,0,%d>' % int(poly)


def _watchdog(seconds, what):
    """A multi-rank run that stops making progress (a peer died, a collective never completes)
    must end by itself: exit non-zero with a message instead of sitting until the driver's limit."""
    import threading

    def bark():
        sys.stderr.write(f'bench.py: {what} made no progress for {seconds} s -- giving up\n')
        sys.stderr.flush()
        os._exit(3)
    t = threading.Timer(seconds, bark)
    t.daemon = True
    t.start()
    return t


def run_b200(args):
    import torch
    import torch.distributed as dist
    from rayoptics_b200 import _abi, table as T, engine as E, analyses as A, parallel as P

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py --impl b200 needs a CUDA device'
    torch.cuda.set_device(local)
    dog = None
    if world > 1:
        import datetime
        dog = _watchdog(600, f'rank {rank} of {world}')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local),
                                timeout=datetime.timedelta(seconds=180))   # fail fast, never hang
    dev = torch.device('cuda', local)
    _abi.load_library()

    opm = load_model(args.model)
    tab = T.SurfaceTable.from_model(opm.seq_model, device=local)
    grid = E.grid_for_model(opm, tab, args.num)
    shard = args.mode == 'shard'
    c0, c1 = P.shard_chunks(grid.n_chunks, rank, world) if shard else (0, grid.n_chunks)
    balance = None
    if shard and world > 1:
        # equal-length ranges leave the ranks with the cheap (clipped) fields idle: one
        # summary-only pass of the equal split gives per-tile costs, the timed steps use ranges
        # of equal WORK (parallel.shard_chunks_weighted).  Outside every timed region.
        r0 = E.trace_grid(tab, grid, c0, c1, outputs=())
        w = P.weights_from_summary(P.gather_summaries(r0.summary))
        equal = (c0, c1)
        c0, c1 = P.shard_chunks_weighted(grid.chunks_per_tile, w, rank, world)
        balance = {'equal_length_range': list(equal), 'equal_work_range': [c0, c1],
                   'tile_weight_min_max': [float(w.min()), float(w.max())]}
    n_mine = grid.rays_in_chunks(c0, c1)             # rays this rank traces per step
    first = grid.first_ray_of_chunk(c0)
    n_job = grid.n_rays if shard else world*grid.n_rays
    res = E.BundleResult(n_mine, tab.n_ifc, dev, E.GRID_OUTPUTS)

    def trace():
        return E.trace_grid(tab, grid, c0, c1, res=res)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    n_warm = max(args.warmup, 3)
    for _ in range(n_warm):             # W warm-up steps: SAME count on every rank (each
        r = trace()                     # step holds a collective)
        if world > 1:
            P.gather_summaries(r.summary)
    torch.cuda.synchronize()
    step_est = None
    t_w, extra = time.perf_counter(), 0
    while time.perf_counter() - t_w < 0.7:
        trace()                             # collective-free extra warm-up, long enough for the
        extra += 1                          # clocks to ramp and nvidia-smi to sample under load
        if extra % 16 == 0 or n_mine > (1 << 24):
            torch.cuda.synchronize()
    barrier()
    # ---- the dominant kernel on its own (roofline): trace + its spot-sum reduction, CUDA events
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
    for a, b in kev:
        a.record()
        trace()
        b.record()
    torch.cuda.synchronize()
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))

    # ---- one step = trace + reduction (+ all-gather + combine when world > 1), captured once as a
    # CUDA graph and replayed K times: the host only issues one graph launch per step, so a busy
    # host (these boxes share their cores between tenants) cannot stretch the device timeline
    launches_per_step = None
    graph = None
    # single GPU only: measured this round (6.2e9 rays/s, profiles/r02k).  With NCCL in the step the
    # capture worked at N=2 and hung at N=4 on the one box it was tried on (NOTES_r02.md), so N > 1
    # keeps the eager loop, whose collective pattern is the one the round-1 scaling run used.
    if not args.no_graph and world == 1:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):                       # same count on every rank (collectives)
                    r = trace()
                    if world > 1:
                        P.gather_summaries(r.summary)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            l0 = E.launch_count()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                r = trace()
                combined = P.gather_summaries(r.summary) if world > 1 else r.summary
            launches_per_step = E.launch_count() - l0
            graph.replay()
            torch.cuda.synchronize()
        except Exception as e:      # noqa: BLE001 - fall back to the eager loop, say so
            graph, graph_error = None, repr(e)
    launches0 = E.launch_count()
    e_first, e_last = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e_first.record()
    if graph is not None:
        for k in range(args.steps):
            graph.replay()
    else:
        pending, combined, n_gathers = None, None, 0
        if world > 1:
            # spot sums of K consecutive steps share one all-gather: two staging blocks alternate, a
            # block is re-used only after the collective that read it has been waited for
            K = max(1, min(args.gather_every, args.steps))
            n_t = grid.n_tiles
            stage = [torch.empty((K, n_t, E.RT_SUMMARY_DOUBLES), dtype=torch.float64, device=dev)
                     for _ in range(2)]
            which, slot = 0, 0
        for k in range(args.steps):
            trace()
            if world > 1:
                stage[which][slot].copy_(res.summary)
                slot += 1
                if slot == K or k == args.steps - 1:
                    if pending is not None:
                        combined = pending.result()       # [slots * n_tiles, 16]: per-step combined sums
                    pending = P.gather_summaries(stage[which][:slot].reshape(slot*n_t, -1), async_op=True)
                    n_gathers += 1
                    which, slot = 1 - which, 0
        if pending is not None:
            combined = pending.result()
    e_last.record()
    barrier()
    wall = time.perf_counter() - t0
    launches = (launches_per_step*args.steps if graph is not None else E.launch_count() - launches0)
    gather_ok = None
    if world > 1 and combined is not None:
        # every rank holds the same combined sums; the ray counts of the last step add up to the job
        last = combined.reshape(-1, grid.n_tiles, E.RT_SUMMARY_DOUBLES)[-1]
        gather_ok = bool(int(last[:, 0:5].sum().item()) == n_job)
    dev_ms = e_first.elapsed_time(e_last)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, first)
    t = torch.tensor([dev_ms, wall*1e3, kern_ms], dtype=torch.float64, device=dev)
    tmin = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
    dev_ms_max, wall_ms_max = float(t[0]), float(t[1])
    imbalance = {'kernel_ms_max_over_ranks': float(t[2]), 'kernel_ms_min_over_ranks': float(tmin[2])}

    # ---- end to end through the public API, host buffers both sides
    e2e = None
    if not args.no_e2e:
        pinned = {'abr': torch.empty((2, n_mine), dtype=torch.float64).pin_memory()}
        kw = dict(table=tab, pinned=pinned)
        if shard:
            kw['shard'] = (rank, world)
            kw['chunk_range'] = (c0, c1)
        for _ in range(3):
            sd = A.spot_diagram(opm, args.num, **kw)
        barrier()
        t1 = time.perf_counter()
        for _ in range(args.steps):
            sd = A.spot_diagram(opm, args.num, **kw)
            if world > 1 and not shard:
                P.gather_summaries(res.summary)
        barrier()
        e2e_s = time.perf_counter() - t1
        te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {'value': n_job*args.steps/float(te[0]), 'unit': UNIT,
               'h2d_bytes_per_step': int(sd.io_bytes['h2d']),
               'd2h_bytes_per_step': int(sd.io_bytes['d2h']),
               'api': f'rayoptics_b200.analyses.spot_diagram(opt_model, {args.num}): grid description from '
                      'host memory every call (pinned staging, one async copy), chief-ray reference points '
                      'on the device, aberrations into pinned host memory at 16 B/ray (status / failing '
                      'surface in the NaN payloads), per-(field,wvl) statistics'}

    # ---- second regime (reported, not the headline): whole rays written, HBM-bound
    full_ray = None
    if rank == 0 and world == 1 and not args.no_e2e and grid.n_rays*tab.n_ifc*80 < 40e9:
        resf = E.BundleResult(grid.n_rays, tab.n_ifc, dev, ('status', 'n_seg', 'full'))
        for _ in range(3):
            E.trace_grid(tab, grid, res=resf, summary=False)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nrep = 10
        f0.record()
        for _ in range(nrep):
            E.trace_grid(tab, grid, res=resf, summary=False)
        f1.record()
        torch.cuda.synchronize()
        ms = f0.elapsed_time(f1)/nrep
        n_seg = int(resf.n_seg.sum().item())                     # segments actually written
        full_bytes = n_seg*80 + grid.n_rays*8
        full_ray = {'ms_per_step': ms, 'rays_per_s': grid.n_rays/(ms*1e-3),
                    'bytes_per_step': int(full_bytes), 'achieved_gbs': full_bytes/(ms*1e-3)/1e9,
                    'kernel': kernel_name(tab.descs).replace('<0,1', '<2,0'),
                    'note': 'every ray segment [p,d,dst,nrml] of every interface written (80 B each)'}
        del resf
    clocks = sampler.stop() if sampler else None   # window: warm-up + timed steps + e2e steps
    # algorithmic flops of this rank's rays (failing-surface histogram of the run), summed over ranks
    status = res.status.cpu().numpy()
    fail_surf = res.fail_surf.cpu().numpy()
    flops, flops_full_ray = algorithmic_flops(tab.descs, status, fail_surf)
    fl = torch.tensor([flops, float((status == 0).sum()), float(status.size)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(fl, op=dist.ReduceOp.SUM)
    if rank == 0:
        fp64_peak = E.measure_fp64_peak(local)
        bpr = res.bytes_per_ray()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = peaks.get('hbm_gbs', 6650.0)
        traffic, ncu = None, {}
        try:     # dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel
            ncu = json.load(open(os.path.join(ROOT, 'profiles', f'traffic_{args.model}_{args.num}.json')))
            traffic = ncu['dram_bytes_per_launch']
        except Exception:
            pass
        # the dominant kernel of THIS rank: its rays, its launch duration
        ach_tf = flops/(kern_ms*1e-3)/1e12
        ach_gbs = n_mine*bpr/(kern_ms*1e-3)/1e9
        roof = {'bound': 'fp64', 'achieved': ach_tf, 'peak': fp64_peak, 'unit': 'TFLOP/s',
                'frac': ach_tf/fp64_peak if fp64_peak else None,
                'peak_source': 'rt_measure_fp64_peak: DFMA chain microbenchmark on this GPU, this run '
                               '(MEASURED_PEAKS.json holds no fp64 entry)',
                'kernel': kernel_name(tab.descs), 'kernel_ms': kern_ms,
                'rays_per_launch': int(n_mine),
                'algorithmic_flop_per_launch': flops,
                'algorithmic_flop_per_full_ray': flops_full_ray,
                'traffic': traffic, 'traffic_source': ncu.get('source'),
                'pipe_utilisation_ncu': (None if ncu.get('fp64_pipe_pct_of_peak') is None
                                         else ncu['fp64_pipe_pct_of_peak']/100),
                'issue_active_ncu': (None if ncu.get('issue_active_pct') is None
                                     else ncu['issue_active_pct']/100),
                'hbm': {'achieved': ach_gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach_gbs/hbm_peak,
                        'bytes_per_ray': bpr,
                        'peak_source': 'MEASURED_PEAKS.json' if 'hbm_gbs' in peaks
                        else 'B200_PROFILING.md fallback'},
                'why_fp64': 'register-resident trace: no HBM input, 80 B/ray of results; the kernel is bound '
                            'by the fp64 vector pipe / issue (DESIGN.md 5), HBM is the secondary figure'}
        line = {'metric': METRIC, 'value': n_job*args.steps/(dev_ms_max*1e-3), 'unit': UNIT,
                'n_gpus': world, 'steps': args.steps, 'warmup': n_warm, 'extra_warmup_traces': extra,
                'ms_per_step': dev_ms_max/args.steps, 'wall_ms_per_step': wall_ms_max/args.steps,
                'higher_is_better': True, 'scaling': 'strong' if shard else 'weak',
                'vs_baseline': None, 'dtype': 'f64',
                'data': 'synthetic', 'config': config_dict(args, opm, grid, world),
                'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches),
                'step_submission': ('one CUDA graph replay per step (trace, spot-sum reduction'
                                    + (', all-gather, combine' if world > 1 else '') + ' captured once)'
                                    if graph is not None else 'eager launches'),
                'roofline': roof,
                'rank_imbalance': (dict(imbalance, shard_balance=balance) if world > 1 else None),
                'collectives': (None if world == 1 else
                                {'all_gathers_in_timed_region': n_gathers, 'steps_per_all_gather': K,
                                 'payload_bytes_per_rank_per_gather': int(K*grid.n_tiles*E.RT_SUMMARY_DOUBLES*8),
                                 'last_combined_ok': gather_ok}),
                'full_ray_regime': None if full_ray is None else dict(
                    full_ray, frac_of_hbm_peak=full_ray['achieved_gbs']/hbm_peak),
                'rays_ok_frac': float(fl[1]/fl[2])}
        try:      # the same model at a reduced grid against rays traced by the REFERENCE's own grid loop
            line['parity_vs_reference'] = parity_vs_reference_golden(args.model, opm, tab)
        except Exception as e:      # noqa: BLE001 - never lose the bench line over a checker
            line['parity_vs_reference'] = {'error': repr(e)}
        if not args.no_cpu_baseline and world == 1:      # rank 0 at N=1 only
            def gpu_records(r0, r1):
                return {k: getattr(res, k)[..., r0:r1].cpu().numpy()
                        for k in ('p', 'd', 'op', 'abr', 'status', 'fail_surf')}
            line['cpu_baseline'] = cpu_baseline(args, opm, gpu=gpu_records)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if dog is not None:
        dog.cancel()


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
