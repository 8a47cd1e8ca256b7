"""raytrace.install(batched=True): the reference's own analysis classes running on the batched
drivers.

CPU: rayoptics.raytr.analyses.RayFan / RayList / RayGrid (importable) are run on the hybrid
model (oracle/ref_model.py) with their per-ray loops `trace_ray_fan / trace_ray_list /
trace_ray_grid` rebound to rayoptics_b200.trace's batched stand-ins (oracle-fed through the
`tracer=` seam) and must reproduce, bit for bit, what the unpatched reference produced
(tests/golden/vectors/<model>_analyses.npz).  What runs here is the reference's own code, so these
tests need its source tree (oracle/ref_harness.py, B200RT_REF_SRC) and skip without it.
"""
import functools
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_model
from oracle import ref_harness as rh
from rayoptics_b200 import trace as TR
from test_trace_drivers import oracle_tracer

pytestmark = pytest.mark.skipif(not rh.available(), reason='needs the ray-optics source tree (B200RT_REF_SRC)')


@pytest.mark.parametrize('name', ['dblgauss', 'rc', 'telecentric', 'fisheye', 'threemir'])
def test_reference_classes_on_batched_loops(name, monkeypatch):
    from oracle import ref_model
    RT, RA = ref_model.modules()
    for fn in ('trace_ray_fan', 'trace_ray_list', 'trace_ray_grid'):
        monkeypatch.setattr(RA, fn, functools.partial(getattr(TR, 'analyses_' + fn), tracer=oracle_tracer))
    z = np.load(os.path.join(GOLDEN, 'vectors', name + '_analyses.npz'))
    n_fan, n_list, n_grid = (int(x) for x in z['num'])
    opm = load_model(name)
    H = ref_model.HybridModel(opm)
    for ci, (f, wl) in enumerate(z['cases']):
        f, wl = int(f), (None if wl < 0 else float(wl))
        fld = opm.optical_spec.field_of_view.fields[f]
        aim = None if fld.aim_info is None else np.array(fld.aim_info)

        def keep_aim():          # as in make_golden_analyses.py: no re-aiming by the reference
            fld.aim_info = None if aim is None else (float(aim) if aim.ndim == 0 else aim.copy())
            fld.chief_ray = ((None, None, -1.0), None)

        for xy in 'xy':
            keep_aim()
            fan = RA.RayFan(H, f=f, wl=wl, xyfan=xy, num_rays=n_fan)
            assert np.array_equal(np.array([p for p, v in fan.fan], dtype=float).reshape(-1, 2),
                                  z[f'fan{xy}_pupil_{ci}'])
            assert np.array_equal(np.array([v for p, v in fan.fan], dtype=float).reshape(-1, 3),
                                  z[f'fan{xy}_vals_{ci}'])
        keep_aim()
        assert np.array_equal(RA.RayList(H, num_rays=n_list, f=f, wl=wl).ray_abr, z[f'list_abr_{ci}'])
        keep_aim()
        assert np.array_equal(RA.RayGrid(H, f=f, wl=wl, num_rays=n_grid).grid, z[f'grid_{ci}'],
                              equal_nan=True)


@pytest.mark.parametrize('name', ['dblgauss', 'triplet'])
def test_reference_short_lists_on_batched_loops(name, monkeypatch):
    """trace_boundary_rays / trace_astigmatism / trace_ray_list_at_field of the reference with their
    5-ray loops rebound (install(batched=True)): same packages, numbers and DataFrames as unpatched"""
    from oracle import ref_model
    RT, RA = ref_model.modules()
    a, b = load_model(name), load_model(name)
    Ha, Hb = ref_model.HybridModel(a), ref_model.HybridModel(b)
    wvl = a.seq_model.central_wavelength()

    def keep(m):
        for f in m.optical_spec.field_of_view.fields:
            f.chief_ray = ((None, None, -1.0), None)
    keep(a)
    want_rays = RT.trace_boundary_rays(Ha, use_named_tuples=True)
    fa = a.optical_spec.field_of_view.fields[-1]
    want_ast = RT.trace_astigmatism(Ha, fa, wvl, 0.01)
    want_df = RT.trace_ray_list_at_field(Ha, [[0., 0.3], [0.2, -0.5]], fa, wvl, 0.0)
    for fn in ('trace_boundary_rays_at_field', 'trace_astigmatism', 'trace_ray_list_at_field'):
        monkeypatch.setattr(RT, fn, functools.partial(getattr(TR, fn), tracer=oracle_tracer))
    keep(b)
    got_rays = RT.trace_boundary_rays(Hb, use_named_tuples=True)
    fb = b.optical_spec.field_of_view.fields[-1]
    assert RT.trace_astigmatism(Hb, fb, wvl, 0.01) == want_ast
    got_df = RT.trace_ray_list_at_field(Hb, [[0., 0.3], [0.2, -0.5]], fb, wvl, 0.0)
    for fw, fg in zip(want_rays, got_rays):
        assert len(fw) == len(fg) == 5
        for pw, pg in zip(fw, fg):
            assert len(pw.ray) == len(pg.ray) and pw.op == pg.op
            for sw, sg in zip(pw.ray, pg.ray):
                assert np.array_equal(sw.p, sg.p) and np.array_equal(sw.d, sg.d) and sw.dst == sg.dst
    for x, y in zip(a.optical_spec.field_of_view.fields, b.optical_spec.field_of_view.fields):
        assert list(x.pupil_rays) == list(y.pupil_rays) == ['00', '+X', '-X', '+Y', '-Y']
    for dw, dg in zip(want_df, got_df):
        assert list(dw.columns) == list(dg.columns) and len(dw) == len(dg)
        for col in dw.columns:
            for u, v in zip(dw[col], dg[col]):
                assert np.array_equal(np.asarray(u), np.asarray(v))


def test_install_batched_rebinds_and_restores():
    from oracle import ref_model
    from rayoptics_b200 import raytrace as B
    RT, RA = ref_model.modules()
    import rayoptics.raytr.raytrace as rt
    orig = (rt.trace, rt.trace_raw, RT.trace_fan, RT.trace_grid, RA.trace_ray_fan, RA.trace_ray_list,
            RA.trace_ray_grid)
    B.install(batched=True)
    try:
        assert rt.trace is B.trace and RA.trace_ray_grid is not orig[6] and RT.trace_fan is not orig[2]
        assert RA.trace_ray_fan.__wrapped__ is orig[4]
    finally:
        B.uninstall()
    assert (rt.trace, rt.trace_raw, RT.trace_fan, RT.trace_grid, RA.trace_ray_fan, RA.trace_ray_list,
            RA.trace_ray_grid) == orig
