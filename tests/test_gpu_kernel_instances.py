"""Every compiled trace-kernel instance of libb200rt.so against the oracle.

``MATRIX`` lists launches -- a fixture, a call, and the template instance the call must reach --
that together reach all 38 ``k_trace_bundle`` / ``k_trace_bundle_lean`` / ``k_trace_grid`` /
``k_trace_grid_lean`` instances.  Each instance has its own register allocation, spill code and
shared-memory layout, so each is run and its every output compared with the oracle bit for bit
(OPD: 1e-12 mm, the bar of DESIGN §3.4; spot sums: tests/test_gpu_spot_sums.py's checks).

Which instance a call reaches is decided in ``rt_table_create`` / ``rt_trace_bundle`` /
``rt_trace_grid``; ``expected_instance`` restates that rule:
- a table is lean when no interface has a transform, aperture list, phase element or thin lens
  and its plan (LeanSurf 112 B per interface + LeanIdx 32 B per (wavelength, interface), plus
  LeanPoly 336 B per interface for a polynomial system) fits in RT_MAX_STAGE_BYTES minus the
  spot-sum accumulators, 174 080 B; B200RT_NO_LEAN forces the general kernels;
- POLY: any profile beyond Conic; STAGE: n_ifc * (640 + 8 * n_wvl) <= 174 080;
- bundles: OUT = 2 with whole rays, 1 when normals / dst are written, 0 otherwise;
- grids: the lean kernels need a lean table and an EPD pupil; WAVE (the opd output) runs with
  OUT 0 only.
A CPU test checks that the matrix names exactly the instances ``nm`` finds in the library and
that the rule gives each entry's instance; on the GPU, torch.profiler records the kernel each
launch ran.

The long systems are committed models whose last air gap is split into equal gaps by planar
dummy interfaces (``LongSeq``), at 3 wavelengths:
- cellphone, 320 interfaces: the polynomial lean plan exactly at the limit (320 * 544 B); with
  spot sums the launch uses 204 800 B of shared memory;
- cellphone, 321 interfaces: the plan overflows -> general, unstaged kernels;
- dblgauss, 262 / 263 interfaces, general kernels: the last staged table (173 968 B) and the
  first unstaged one.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import load_model, seeded_bundle
from rayoptics_b200 import _abi, engine as E, table as T, model as M, waveabr as W
from test_gpu_spot_sums import DRYRUN, check_launch

STAGE_LIMIT = 200*1024 - 15*256*8                  # RT_MAX_STAGE_BYTES - RT_ACC_BYTES
LEAN_SURF, LEAN_IDX, LEAN_POLY = 112, 32, 336     # sizeof LeanSurf / LeanIdx / LeanPoly
OPD_TOL_MM = 1e-12


# ----------------------------------------------------------------- fixtures
class LongSeq:
    """A sequential model's path with its last air gap split into equal gaps by planar dummy
    interfaces, ``n_ifc`` interfaces in all (what SurfaceTable.from_model needs of a model)."""

    def __init__(self, seq_model, n_ifc):
        self.sm, self.wvlns = seq_model, list(seq_model.wvlns)
        self.extra = n_ifc - len(seq_model.ifcs)

    def central_wavelength(self):
        return self.sm.central_wavelength()

    def path(self, wl=None):
        segs = list(self.sm.path(wl))
        ifc, gap, (rt, t), n, z = segs[-2]
        assert np.array_equal(rt, np.identity(3)) and t[0] == 0.0 and t[1] == 0.0
        k = self.extra + 1
        step = (np.identity(3), np.array([0.0, 0.0, t[2]/k]))
        dummies = [(M.Surface('split', interact_mode='dummy', max_aperture=1.0e3), gap, step, n, z)
                   for _ in range(self.extra)]
        return iter(segs[:-2] + [(ifc, gap, step, n, z)] + dummies + segs[-1:])


FIXTURES = {       # name: (model, interfaces (None: as committed), B200RT_NO_LEAN)
    'dblgauss': ('dblgauss', None, False),
    'dblgauss_general': ('dblgauss', None, True),
    'cellphone': ('cellphone', None, False),
    'exotic': ('exotic', None, False),
    'cellphone_320': ('cellphone', 320, False),
    'cellphone_321': ('cellphone', 321, False),
    'dblgauss_262_general': ('dblgauss', 262, True),
    'dblgauss_263_general': ('dblgauss', 263, True),
}


def fixture_seq(name):
    model, n_ifc, _ = FIXTURES[name]
    opm = load_model(model)
    return opm, (opm.seq_model if n_ifc is None else LongSeq(opm.seq_model, n_ifc))


# ----------------------------------------------------------------- the selection rule
def table_kind(descs, n_wvl, no_lean):
    """(lean, poly, stage) as rt_table_create decides them"""
    n = len(descs)
    poly = any(d.profile > _abi.PROFILE_IDS['Conic'] for d in descs)
    stage = n*(C.sizeof(_abi.rt_surface_desc) + 8*n_wvl) <= STAGE_LIMIT
    plan = n*(LEAN_SURF + LEAN_IDX*n_wvl + (LEAN_POLY if poly else 0))
    lean = (not no_lean and plan <= STAGE_LIMIT and
            all(d.has_tfrm == 0 and d.n_apertures == 0 and d.phase_kind == 0 and
                d.profile != _abi.PROFILE_IDS['ThinLens'] for d in descs))
    return lean, poly, stage


def expected_instance(kind, call):
    lean, poly, stage = kind
    b = lambda v: str(int(bool(v)))                 # noqa: E731
    out = call.get('out', 0)
    if call['call'] == 'bundle':
        return (f'k_trace_bundle_lean<{out},{b(poly)}>' if lean
                else f'k_trace_bundle<{b(out == 2)},{b(stage)}>')
    s, wave = call.get('summary', False), call.get('wave', False)
    if wave:
        assert out == 0
    if lean:                                        # all grids here have an EPD pupil
        return f'k_trace_grid_lean<{out},{b(s)},{b(wave)},{b(poly)}>'
    return f'k_trace_grid<{b(out == 2)},{b(s)},{b(stage)},{b(wave)}>'


def bundle(out, n=4000):
    return dict(call='bundle', out=out, n=n)


def grid(out=0, summary=False, wave=False, num=33, one_tile=False):
    return dict(call='grid', out=out, summary=summary, wave=wave, num=num, one_tile=one_tile)


MATRIX = [   # (fixture, call, instance it reaches)
    ('dblgauss', bundle(0), 'k_trace_bundle_lean<0,0>'),
    ('dblgauss', bundle(1), 'k_trace_bundle_lean<1,0>'),
    ('dblgauss', bundle(2), 'k_trace_bundle_lean<2,0>'),
    ('cellphone', bundle(0), 'k_trace_bundle_lean<0,1>'),
    ('cellphone', bundle(2), 'k_trace_bundle_lean<2,1>'),
    ('cellphone_320', bundle(1), 'k_trace_bundle_lean<1,1>'),
    ('cellphone_320', bundle(2, 2000), 'k_trace_bundle_lean<2,1>'),
    ('exotic', bundle(1), 'k_trace_bundle<0,1>'),
    ('exotic', bundle(2), 'k_trace_bundle<1,1>'),
    ('dblgauss_262_general', bundle(2, 2000), 'k_trace_bundle<1,1>'),
    ('dblgauss_263_general', bundle(1), 'k_trace_bundle<0,0>'),
    ('dblgauss_263_general', bundle(2, 2000), 'k_trace_bundle<1,0>'),
    ('cellphone_321', bundle(0), 'k_trace_bundle<0,0>'),
    ('cellphone_321', bundle(2, 2000), 'k_trace_bundle<1,0>'),
    # lean grids, conic
    ('dblgauss', grid(0), 'k_trace_grid_lean<0,0,0,0>'),
    ('dblgauss', grid(0, True, num=47), 'k_trace_grid_lean<0,1,0,0>'),
    ('dblgauss', grid(1), 'k_trace_grid_lean<1,0,0,0>'),
    ('dblgauss', grid(1, True), 'k_trace_grid_lean<1,1,0,0>'),
    ('dblgauss', grid(2, num=20), 'k_trace_grid_lean<2,0,0,0>'),
    ('dblgauss', grid(2, True, num=20), 'k_trace_grid_lean<2,1,0,0>'),
    ('dblgauss', grid(0, False, True), 'k_trace_grid_lean<0,0,1,0>'),
    ('dblgauss', grid(0, True, True, num=47), 'k_trace_grid_lean<0,1,1,0>'),
    # lean grids, polynomial
    ('cellphone', grid(0), 'k_trace_grid_lean<0,0,0,1>'),
    ('cellphone', grid(0, True), 'k_trace_grid_lean<0,1,0,1>'),
    ('cellphone_320', grid(0, True, num=20), 'k_trace_grid_lean<0,1,0,1>'),
    ('cellphone', grid(1), 'k_trace_grid_lean<1,0,0,1>'),
    ('cellphone_320', grid(1, True, num=20), 'k_trace_grid_lean<1,1,0,1>'),
    ('cellphone', grid(2, num=17), 'k_trace_grid_lean<2,0,0,1>'),
    ('cellphone_320', grid(2, True, num=41, one_tile=True), 'k_trace_grid_lean<2,1,0,1>'),
    ('cellphone', grid(0, False, True), 'k_trace_grid_lean<0,0,1,1>'),
    ('cellphone_320', grid(0, True, True, num=20), 'k_trace_grid_lean<0,1,1,1>'),
    # general grids, staged
    ('exotic', grid(0), 'k_trace_grid<0,0,1,0>'),
    ('exotic', grid(1, True, num=47), 'k_trace_grid<0,1,1,0>'),
    ('exotic', grid(2, num=20), 'k_trace_grid<1,0,1,0>'),
    ('exotic', grid(2, True, num=20), 'k_trace_grid<1,1,1,0>'),
    ('dblgauss_general', grid(0, False, True), 'k_trace_grid<0,0,1,1>'),
    ('dblgauss_general', grid(0, True, True, num=47), 'k_trace_grid<0,1,1,1>'),
    ('dblgauss_262_general', grid(0, True, num=20), 'k_trace_grid<0,1,1,0>'),
    # general grids, unstaged
    ('dblgauss_263_general', grid(0, True, num=20), 'k_trace_grid<0,1,0,0>'),
    ('cellphone_321', grid(0, num=20), 'k_trace_grid<0,0,0,0>'),
    ('cellphone_321', grid(1, True, num=20), 'k_trace_grid<0,1,0,0>'),
    ('cellphone_321', grid(2, num=33, one_tile=True), 'k_trace_grid<1,0,0,0>'),
    ('cellphone_321', grid(2, True, num=41, one_tile=True), 'k_trace_grid<1,1,0,0>'),
    ('cellphone_321', grid(0, False, True, num=20), 'k_trace_grid<0,0,0,1>'),
    ('cellphone_321', grid(0, True, True, num=33), 'k_trace_grid<0,1,0,1>'),
]


def entry_id(entry):
    fx, call, inst = entry
    keys = ''.join(f'-{k}{int(v)}' for k, v in call.items() if k in ('out', 'summary', 'wave'))
    return f'{inst}-{fx}-{call["call"]}{keys}-n{call.get("num", call.get("n"))}'


def canonical(name):
    """'void k_trace_grid<false, true, true, false>(...)' -> 'k_trace_grid<0,1,1,0>' (or None)"""
    m = re.search(r'\b(k_trace_(?:bundle|grid)(?:_lean)?)<([^<>]*)>', name)
    if not m:
        return None
    args = [a.strip() for a in m.group(2).split(',')]
    return m.group(1) + '<' + ','.join({'true': '1', 'false': '0'}.get(a, a) for a in args) + '>'


# ----------------------------------------------------------------- CPU
def test_matrix_covers_every_compiled_instance():
    """the instances nm lists in the built library are exactly the matrix's"""
    out = subprocess.run(['nm', '-C', '--defined-only', _abi.lib_path()], check=True,
                         capture_output=True, text=True).stdout
    compiled = {canonical(line) for line in out.splitlines()} - {None}
    assert len(compiled) == 38
    assert compiled == {inst for _, _, inst in MATRIX}


@pytest.mark.parametrize('fixture', sorted(FIXTURES))
def test_selection_rule_gives_each_entrys_instance(fixture):
    """the rule restated from rt_table_create / rt_trace_* gives the instance every entry names;
    the long fixtures sit where the matrix says (plan / table sizes at the limits)"""
    opm, seq = fixture_seq(fixture)
    descs, n_by_wvl, _ = T.describe_model(seq)
    n_wvl, n = n_by_wvl.shape
    kind = table_kind(descs, n_wvl, FIXTURES[fixture][2])
    sizes = {'cellphone_320': (320, 320*544, True), 'cellphone_321': (321, 321*544, False)}
    if fixture in sizes:
        n_want, plan, lean = sizes[fixture]
        assert n == n_want and n_wvl == 3 and kind[0] == lean and kind[1]
        if lean:        # with spot sums the launch asks for all of RT_MAX_STAGE_BYTES
            assert plan == STAGE_LIMIT and plan + 15*256*8 == 204800
        else:
            assert plan == STAGE_LIMIT + 544 and not kind[2]
    if fixture == 'dblgauss_262_general':
        assert n == 262 and n*(640 + 8*3) == 173968 and kind == (False, False, True)
    if fixture == 'dblgauss_263_general':
        assert n == 263 and kind == (False, False, False)
    if fixture == 'cellphone_321':
        d = descs[n - 2]            # the last interface before the image: OPD is allowed
        assert d.has_tfrm == 0 and d.t[0] == 0.0 and d.t[1] == 0.0 and d.mode == _abi.MODE_IDS['dummy']
    entries = [e for e in MATRIX if e[0] == fixture]
    assert entries
    for _, call, inst in entries:
        assert expected_instance(kind, call) == inst, (fixture, call)


# ----------------------------------------------------------------- GPU
_TABLES = {}


def get_table(fixture):
    if fixture not in _TABLES:
        opm, seq = fixture_seq(fixture)
        no_lean = FIXTURES[fixture][2]
        old = os.environ.pop('B200RT_NO_LEAN', None)
        try:
            if no_lean:
                os.environ['B200RT_NO_LEAN'] = '1'
            tab = T.SurfaceTable.from_model(seq, device=0)
        finally:
            os.environ.pop('B200RT_NO_LEAN', None)
            if old is not None:
                os.environ['B200RT_NO_LEAN'] = old
        _TABLES[fixture] = (opm, tab)
    return _TABLES[fixture]


def profiled(fn):
    """fn() under torch.profiler; returns (result, names of the trace kernels it launched)"""
    if DRYRUN:
        return fn(), None
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [canonical(e.name) for e in prof.events()]
    return res, [n for n in names if n]


def np_(t):
    return None if t is None else t.detach().cpu().numpy()


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def check_rays(r, ref, opd_ref=None):
    """every per-ray output the launch wrote against the oracle"""
    assert same(np_(r.status), ref['status'])
    assert same(np_(r.fail_surf), ref['fail_surf'])
    assert same(np_(r.op), ref['op'])
    assert same(np_(r.p), ref['last'][0:3]) and same(np_(r.d), ref['last'][3:6])
    if r.dst is not None:
        assert same(np_(r.dst), ref['last'][6])
    if r.nrml is not None:
        assert same(np_(r.nrml), ref['last'][7:10])
    if r.n_seg is not None:
        assert same(np_(r.n_seg), ref['n_seg'])
    if r.full is not None:
        assert same(np_(r.full), ref['full'])
    if r.abr is not None:
        assert same(np_(r.abr), ref['abr'])
    if r.opd is not None:
        opd, ok = np_(r.opd), ref['status'] == 0
        assert same(np.isnan(opd), np.isnan(opd_ref)) and np.isnan(opd[~ok]).all()
        assert np.abs(opd[ok] - opd_ref[ok]).max(initial=0.0) <= OPD_TOL_MM


def run_bundle(oracle, opm, tab, call):
    rng = np.random.default_rng(17)
    p0, d0, wv = seeded_bundle(opm, call['n'], rng)
    case = dict(first_surf=1, last_surf=tab.n_ifc - 2, check_apertures=True)
    outputs = ('p', 'd', 'op', 'status', 'fail_surf', 'n_seg') if call['out'] == 0 else E.BUNDLE_OUTPUTS
    r, names = profiled(lambda: E.trace_bundle(tab, p0, d0, wvl_idx=wv, full=call['out'] == 2,
                                                 outputs=outputs, **case))
    ref = oracle.trace_bundle(tab.descs, tab.n_by_wvl, p0, d0, wv, _abi.make_opts(**case),
                              want_full=call['out'] == 2, n_threads=8, wvls=tab.wvls)
    check_rays(r, ref)
    assert (ref['status'] == 0).sum() > call['n']//10
    return names


def run_grid(oracle, opm, tab, call):
    osp, sm = opm.optical_spec, opm.seq_model
    fields, wvls = list(osp.field_of_view.fields), list(sm.wvlns)
    if call['one_tile']:
        fields, wvls = fields[-1:], wvls[:1]
    num = call['num']
    if call['wave']:
        # wavefront records of the committed model: an input the kernel and the oracle share
        short = T.SurfaceTable.from_model(sm, device=0)
        wave, ref_img, _ = W.setup_tiles(opm, short, fields, wvls, 0.0)
        recs, eprad, z_pupil = osp.grid_fields(fields)
        xs = E.accumulated_steps(-1.0, 1.0, num)
        g = E.PupilGrid(recs, [tab.wvl_index(w) for w in wvls], xs, xs, eprad, z_pupil,
                        ref_img=ref_img, flip_z_dir=sm.z_dir[0], wave=wave, device=0)
    else:
        g = E.grid_for_model(opm, tab, num, fields=fields, wvls=wvls)
    outputs = E.GRID_OUTPUTS + (('opd',) if call['wave'] else ())
    if call['out'] >= 1:
        outputs += ('nrml', 'dst', 'n_seg')
    torch.cuda.synchronize()
    r, names = profiled(lambda: E.trace_grid(tab, g, outputs=outputs, full=call['out'] == 2,
                                             summary=call['summary']))
    opts = _abi.make_opts(first_surf=1, last_surf=tab.n_ifc - 2, check_apertures=True)
    spec = g.c_spec()
    ref = oracle.trace_grid(spec, tab.descs, tab.n_by_wvl, 0, g.n_rays, opts, n_threads=8,
                            wvls=tab.wvls)
    if call['out'] >= 1:
        p, d, wv, _ = oracle.grid_start_rays(spec, 0, g.n_rays)
        b = oracle.trace_bundle(tab.descs, tab.n_by_wvl, p, d, wv, opts,
                                want_full=call['out'] == 2, n_threads=8, wvls=tab.wvls)
        assert same(b['last'], ref['last']) and same(b['status'], ref['status'])
        ref['n_seg'], ref['full'] = b['n_seg'], b['full']
    check_rays(r, ref, ref['opd'])
    ok = ref['status'] == 0
    assert ok.sum() > g.n_rays//5
    if call['summary']:
        check_launch(np_(r.summary), g, 0, g.n_chunks, np_(r.abr), np_(r.op), np_(r.status))
    else:
        assert r.summary is None
    return names


@pytest.mark.gpu
@pytest.mark.parametrize('entry', MATRIX, ids=[entry_id(e) for e in MATRIX])
def test_instance_matches_oracle(oracle, entry):
    fixture, call, inst = entry
    opm, tab = get_table(fixture)
    run = run_bundle if call['call'] == 'bundle' else run_grid
    names = run(oracle, opm, tab, call)
    if names is not None:
        assert names == [inst]
