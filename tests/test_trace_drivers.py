"""Host logic of rayoptics_b200/trace.py, SequentialModel.trace_fan/trace_grid/
trace_wavefront and analyses.Ray (the reference's raytr/trace.py:159-219,537-624,
seq/sequential.py:1006-1120, raytr/analyses.py:46-118).

CPU: the `tracer=` seam is fed by the oracle, the expected values come from the
reference's own trace_raw on start rays built by opticalspec.ray_start_from_osp
(stored under tests/golden/reference/ by tests/refdata.py; whole ray packages as digest())
and from the golden OPD vectors.  The GPU run of the
same calls is in tests/test_zz_gpu_additions.py.
"""
import os

import numpy as np
import pytest

from conftest import load_model
from rayoptics_b200 import _abi, engine as E, table as T, trace as TR, waveabr as W
from rayoptics_b200 import analyses as A
from refdata import digest, lens_files, ref  # noqa: F401


def oracle_tracer(opt_model, table, fld, wvl, px, py, apply_vignetting, trace_kwargs):
    """tracer= seam: start rays + trace by oracle/rt_oracle.c (test infrastructure)."""
    from oracle import rt_oracle
    osp, sm = opt_model.optical_spec, opt_model.seq_model
    descs, n_by_wvl, wvls = T.describe_model(sm)
    recs, eprad, z_pupil = osp.grid_fields([fld])
    spec = E.PupilGridSpec(recs, [sm.index_for_wavelength(wvl)], px, py, eprad, z_pupil,
                           apply_vignetting=apply_vignetting, flip_z_dir=sm.z_dir[0], paired=True)
    p, d, wv, _ = rt_oracle.grid_start_rays(spec.c_spec(), 0, spec.n_rays)
    kw = {k: v for k, v in trace_kwargs.items() if k in TR._TRACE_RAW_KEYS}
    kw.setdefault('check_apertures', False)
    kw.setdefault('first_surf', 1)
    kw.setdefault('last_surf', len(descs) - 2)
    if osp.field_of_view.is_wide_angle:       # engine.trace_grid does this for RT_PUPIL_WIDE grids
        kw['intersect_obj'] = False
    r = rt_oracle.trace_bundle(descs, n_by_wvl, p, d, wv, _abi.make_opts(**kw), want_full=True,
                               wvls=wvls)
    return r


def ref_pkg(opm, fld, wvl, pupil, apply_vignetting=True, **kw):
    from oracle import ref_harness as rh
    osp, sm = opm.optical_spec, opm.seq_model
    vp = fld.apply_vignetting(np.array(pupil)) if apply_vignetting else np.array(pupil)
    pt0, dir0 = osp.ray_start_from_osp(vp, fld)
    if dir0[2]*sm.z_dir[0] < 0:
        dir0 = -dir0
    kw.setdefault('first_surf', 1)
    kw.setdefault('last_surf', sm.get_num_surfaces() - 2)
    return rh.ref_trace(rh.ref_path(sm, wvl), pt0, dir0, wvl, **kw)


def ref_pkg_digest(*args, **kw):
    """ref_pkg with the segments [n_seg, 10] as digest()"""
    r = ref_pkg(*args, **kw)
    return dict(r, ray=digest(r['ray']))


def pkg_digest(pkg):
    """digest() of a ray package's segments (p, d, dst, nrml) and optical path"""
    return digest([[tuple(seg)[:4] for seg in pkg[0]], pkg[1]])


def assert_pkg_equals(pkg, ref):
    ray, op, _ = pkg
    assert len(ray) == ref['n_seg']
    if isinstance(ref['ray'], str):             # stored as digest() of the [n_seg, 10] segments
        assert digest([np.concatenate([seg[0], seg[1], [seg[2]], seg[3]]) for seg in ray]) == ref['ray']
    else:
        for k, seg in enumerate(ray):
            assert np.array_equal(seg[0], ref['ray'][k, 0:3]) and np.array_equal(seg[1], ref['ray'][k, 3:6])
            assert seg[2] == ref['ray'][k, 6] and np.array_equal(seg[3], ref['ray'][k, 7:10])
    assert op == ref['op']


def test_trace_fan_and_grid_against_reference_rays(ref):
    opm = load_model('dblgauss')
    osp = opm.optical_spec
    fld, wvl = osp.field_of_view.fields[2], 486.1
    fan_def = [np.array([0., -1.]), np.array([0., 1.]), 9]
    fan = TR.trace_fan(opm, fan_def, fld, wvl, 0.0, tracer=oracle_tracer)
    t = E.accumulated_steps(-1.0, 1.0, 9)
    # what is recorded are the accumulated pupil values AFTER Field.apply_vignetting (the
    # reference's trace_base vignettes its ndarray argument in place)
    assert [f[0][1] for f in fan] == [fld.apply_vignetting(np.array([0., v]))[1] for v in t]
    for (pupil, pkg), v in zip(fan, t):
        assert_pkg_equals(pkg, ref(lambda: ref_pkg_digest(opm, fld, wvl, [0., v])))
    # grid: check_apertures forced on, failed rays -> None entries, x outer / y inner
    grid_def = [np.array([-1., -1.]), np.array([1., 1.]), 7]
    seen = []
    g = TR.trace_grid(opm, grid_def, fld, wvl, 0.0, tracer=oracle_tracer, form='list',
                      img_filter=lambda p, pkg: seen.append((tuple(p), pkg)) or (None if pkg is None else 1.0),
                      append_if_none=False)
    assert len(seen) == 49
    xs = E.accumulated_steps(-1.0, 1.0, 7)
    vig = lambda a, b: tuple(fld.apply_vignetting(np.array([a, b])))     # noqa: E731
    assert seen[8][0] == vig(xs[1], xs[1]) and seen[6][0] == vig(xs[0], xs[6])
    n_ok = 0
    raw = [[xs[i], xs[j]] for i in range(7) for j in range(7)]
    for (pupil, pkg), p_raw in zip(seen, raw):
        want = ref(lambda: ref_pkg_digest(opm, fld, wvl, p_raw, check_apertures=True))
        assert (pkg is None) == (want['status'] != 0)
        if pkg is not None:
            n_ok += 1
            assert_pkg_equals(pkg, want)
    assert 0 < n_ok < 49 and g.shape == (n_ok,)
    g2 = TR.trace_grid(opm, grid_def, fld, wvl, 0.0, tracer=oracle_tracer)
    assert g2.shape[:2] == (7, 7)


def test_trace_safe_filters_and_errors():
    opm = load_model('dblgauss')
    fld, wvl = opm.optical_spec.field_of_view.fields[0], 587.6
    kw = dict(tracer=oracle_tracer, check_apertures=True)
    ok, bad = np.array([0., 0.5]), np.array([0., 1.3])
    r = TR.trace_safe(opm, ok, fld, wvl, None, None, use_named_tuples=True, **kw)
    assert r.err is None and isinstance(r.pkg, TR.RayPkg) and isinstance(r.pkg.ray[0], TR.RaySeg)
    assert len(r.pkg.ray) == opm.seq_model.get_num_surfaces() and r.pkg.wvl == wvl
    last = TR.trace_safe(opm, ok, fld, wvl, 'last', None, **kw)
    assert len(last.pkg.ray) == 1 and np.array_equal(last.pkg.ray[0][0], r.pkg.ray[-1].p)
    assert TR.trace_safe(opm, ok, fld, wvl, lambda pkg: 42, None, **kw).pkg == 42
    assert TR.trace_safe(opm, bad, fld, wvl, None, None, **kw) == (None, None)
    s = TR.trace_safe(opm, bad, fld, wvl, None, 'summary', **kw)
    assert s.pkg is None and type(s.err).__name__ == 'TraceRayBlockedError' and s.err.ray_pkg is None
    f = TR.trace_safe(opm, bad, fld, wvl, None, 'full', **kw)
    assert isinstance(f.pkg, TR.RayPkg) and f.err.surf == len(f.pkg.ray) - 1 and f.pkg is f.err.ray_pkg
    with pytest.raises(type(f.err)):
        TR.trace_base(opm, bad, fld, wvl, **kw)


def test_sequential_model_drivers_and_ray():
    opm = load_model('dblgauss')
    sm, osp = opm.seq_model, opm.optical_spec
    fod = osp.fod

    def y_abr(p, xy, ray_pkg, fld, wvl, foc):
        return ray_pkg[0][-1][0][xy] - fld.ref_sphere[0][xy]

    fx, fy, (max_rho, max_y), rc = sm.trace_fan(y_abr, 1, 1, num_rays=11, tracer=oracle_tracer)
    assert fx.shape == fy.shape == (3, 11) and max_y > 0 and len(rc) == 3
    assert max_rho == 1.0 - osp.field_of_view.fields[1].vuy          # vignetted pupil coordinates
    assert abs(fy[1, 5]) < 1e-12                    # chief ray of the central wavelength

    def opd(p, wi, ray_pkg, fld, wvl, foc):
        if ray_pkg is None:
            return None
        return W.wave_abr_full_calc(fod, fld, wvl, foc, ray_pkg, fld.chief_ray, fld.ref_sphere)

    grids, _ = sm.trace_grid(opd, 0, wl=587.6, num_rays=9, form='list', append_if_none=False,
                             tracer=oracle_tracer)
    assert len(grids) == 1 and 20 < grids[0].shape[0] < 81 and np.isfinite(grids[0].astype(float)).all()
    wf = sm.trace_wavefront(osp.field_of_view.fields[0], 587.6, 0.0, num_rays=8, tracer=oracle_tracer)
    assert wf.shape == (8, 8, 3) and wf[0, 0, 2] == 0.0 and np.abs(wf[:, :, 2]).max() < 50
    ray = A.Ray(opm, [0., 0.7], f=1, wl=656.3, srf_save='all', tracer=oracle_tracer)
    assert ray.t_abr.shape == (2,) and len(ray.ray_pkg.ray) == sm.get_num_surfaces()
    cr = A.Ray(opm, [0., 0.], f=1, tracer=oracle_tracer)
    assert np.abs(cr.t_abr).max() == 0.0


def oracle_bundle_tracer(opt_model, table, p0, d0, wvl_idx, trace_kwargs):
    from oracle import rt_oracle
    descs, n_by_wvl, wvls = T.describe_model(opt_model.seq_model)
    return rt_oracle.trace_bundle(descs, n_by_wvl, p0, d0, wvl_idx, _abi.make_opts(**trace_kwargs),
                                  want_full=True, wvls=wvls)


def test_trace_list_of_rays(ref):
    from conftest import load_vectors
    from oracle import ref_harness as rh
    opm = load_model('triplet')
    sm = opm.seq_model
    v = load_vectors('triplet')
    idx = np.nonzero(v['case'] == 0)[0][:40]
    rays = [(v['p0'][:, k], v['d0'][:, k], sm.wvlns[v['wvl_idx'][k]]) for k in idx]
    case = dict(v['cases'][0])
    out = A.trace_list_of_rays(opm, rays, rayerr_filter='full', tracer=oracle_bundle_tracer,
                               check_apertures=case['check_apertures'])
    assert len(out) == len(rays)
    n_err = 0
    def ref_trace(pt0, dir0, wvl):
        r = rh.ref_trace(rh.ref_path(sm, wvl), pt0, dir0, wvl, **case)
        return dict(r, ray=digest(r['ray']))
    for (pt0, dir0, wvl), item in zip(rays, out):
        want = ref(lambda: ref_trace(pt0, dir0, wvl))
        if want['status'] == 0:
            assert_pkg_equals(item, want)
        else:
            n_err += 1
            ray, err = item
            assert err.surf == want['fail_surf'] and len(err.ray_pkg[0]) == want['n_seg']
    last = A.trace_list_of_rays(opm, rays, output_filter='last', tracer=oracle_bundle_tracer,
                                check_apertures=case['check_apertures'])
    assert len(last) == len(rays) - n_err and len(last[0]) == 3 and len(last[0][0]) == 4
    assert A.trace_list_of_rays(opm, [], tracer=oracle_bundle_tracer) == []


@pytest.mark.parametrize('name', ['dblgauss', 'rc'])
def test_host_opd_matches_reference(oracle, name):
    """waveabr.wave_abr_full_calc (numpy, for callbacks) against the reference's OPDs"""
    import os
    from conftest import GOLDEN
    z = np.load(os.path.join(GOLDEN, 'vectors', name + '_opd.npz'))
    v = {k: z[k] for k in z.files}
    opm = load_model(name)
    osp, sm = opm.optical_spec, opm.seq_model
    descs, n_by_wvl, _ = T.describe_model(sm)
    n_ifc = len(descs)
    opts = _abi.make_opts(first_surf=1, last_surf=n_ifc - 2, check_apertures=True)
    r = oracle.trace_bundle(descs, n_by_wvl, v['p0'], v['d0'], v['wvl_idx'], opts, want_full=True)
    fields, wvls = osp.field_of_view.fields, sm.wvlns
    checked = 0
    for k in np.nonzero(v['status'] == 0)[0][::7]:
        fi, wi = divmod(int(v['tile'][k]), len(wvls))
        fld, wvl = fields[fi], wvls[wi]
        rs, crp = TR.setup_pupil_coords(opm, fld, wvl, 0.0, tracer=oracle_tracer)
        pkg, err = __import__('rayoptics_b200.raytrace', fromlist=['x']).package_ray(
            list(sm.path(wvl)), r['full'][:, :, k], float(r['op'][k]), 0, -1, n_ifc, wvl)
        got = W.wave_abr_full_calc(osp.fod, fld, wvl, 0.0, pkg, crp, rs)
        assert got == v['opd'][k]
        checked += 1
    assert checked > 20


def oracle_bundle_fn(opm):
    from oracle import rt_oracle
    descs, n_by_wvl, wvls = T.describe_model(opm.seq_model)

    def fn(p0, d0, wvl):
        w = np.full(p0.shape[1], opm.seq_model.index_for_wavelength(wvl), dtype=np.int32)
        r = rt_oracle.trace_bundle(descs, n_by_wvl, p0, d0, w,
                                   _abi.make_opts(first_surf=1, last_surf=len(descs) - 2),
                                   want_full=True, wvls=wvls)
        return r['full'], r['n_seg']
    return fn


@pytest.mark.parametrize('name', ['triplet', 'dblgauss', 'evenasph'])
def test_batched_aiming_and_apertures(name):
    """aim points: the stored ones of the reference's .roa files (its iterate_ray) where the
    model came from a .roa, the per-ray Newton iteration otherwise; apertures: the per-ray
    version on the same rays"""
    from rayoptics_b200 import vigcalc as V
    opm = load_model(name)
    stored = [None if f.aim_info is None else np.array(f.aim_info, dtype=float)
              for f in opm.optical_spec.field_of_view.fields]
    stored_ap = [ifc.max_aperture for ifc in opm.seq_model.ifcs]
    fn = oracle_bundle_fn(opm)
    aims = V.aim_all_fields_batched(opm, fn)
    for a, s in zip(aims, stored):
        if s is not None:
            assert np.abs(a - s).max() < 1e-7   # .roa aim points: scipy newton at its default tol (1.5e-8)
    V.set_clear_apertures_batched(opm, fn)
    got_ap = [ifc.max_aperture for ifc in opm.seq_model.ifcs]
    np.testing.assert_allclose(got_ap[1:-1], stored_ap[1:-1], rtol=1e-6)


def test_set_vig_grazes_the_limiting_apertures():
    """set_vig (raytr/vigcalc.py:83-90,227-342): after it, every boundary ray of every field
    passes with clipping and touches a clear aperture (the limiting one) to the secant
    tolerance; on axis nothing is vignetted (apertures were set from the same rays)."""
    from rayoptics_b200 import vigcalc as V
    opm = load_model('dblgauss')
    osp, sm = opm.optical_spec, opm.seq_model
    fields = osp.field_of_view.fields
    stored = [(f.vux, f.vlx, f.vuy, f.vly) for f in fields]
    for f in fields:
        f.vux = f.vlx = f.vuy = f.vly = 0.0
    V.set_vig(opm, tracer=oracle_tracer)
    got = [(f.vux, f.vlx, f.vuy, f.vly) for f in fields]
    assert max(abs(v) for v in got[0]) < 1e-5               # axial bundle fills the stop
    # the fixture's apertures were set to pass the rays with VUY/VLY = .2/.25 and .4/.4, so
    # the apertures cannot vignette more than that
    for g, s in zip(got[1:], stored[1:]):
        assert -1e-4 <= g[2] <= s[2] + 1e-4 and -1e-4 <= g[3] <= s[3] + 1e-4 and 0 <= g[0] < 0.5
    wvl = osp.spectral_region.central_wvl
    for f in fields:
        for pr in osp.pupil.pupil_rays[1:]:
            res = TR.trace_safe(opm, np.array(pr), f, wvl, None, 'full', tracer=oracle_tracer,
                                check_apertures=True, pt_inside_fuzz=2e-4)
            assert res.err is None                          # with the new factors the ray passes
            slack = min(ifc.max_aperture - np.hypot(seg[0][0], seg[0][1])
                        for ifc, seg in list(zip(sm.ifcs, res.pkg[0]))[1:-1])
            assert -2e-4 < slack < 2e-3                     # ... and grazes the limiting aperture


def test_trace_ray_and_boundary_rays():
    opm = load_model('triplet')
    osp = opm.optical_spec
    fld, wvl = osp.field_of_view.fields[-1], opm.seq_model.central_wavelength()
    rr = TR.trace_ray(opm, [0., 0.5], fld, wvl, tracer=oracle_tracer)
    assert rr.err is None and isinstance(rr.pkg, TR.RayPkg) and isinstance(rr.pkg.ray[0], TR.RaySeg)
    rayset = TR.trace_boundary_rays(opm, tracer=oracle_tracer, use_named_tuples=True)
    assert len(rayset) == len(osp.field_of_view.fields) and all(len(r) == 5 for r in rayset)
    assert set(fld.pupil_rays) == {'00', '+X', '-X', '+Y', '-Y'}
    # the chief ray of the set is the (0, 0) ray setup_pupil_coords traced
    assert np.array_equal(rayset[-1][0].ray[-1].p, fld.chief_ray[0].ray[-1][0])
    # the clear apertures of the .roa model are the max heights of exactly these rays
    hts = [max(np.hypot(r.ray[2].p[0], r.ray[2].p[1]) for rim in rayset for r in rim)]
    assert hts[0] == pytest.approx(opm.seq_model.ifcs[2].max_aperture, rel=1e-6)


def test_iterate_ray_is_the_references(ref):
    """vigcalc.iterate_ray against the reference's iterate_ray, whose source text is executed
    from the reference tree (its module cannot be imported: opticalglass is absent) on the
    reference's own trace_raw."""
    import ast
    import logging
    import warnings
    from scipy.optimize import newton, fsolve
    from oracle import ref_harness as rh
    from rayoptics_b200 import vigcalc as V

    def reference_iterate_ray(name, fi):
        R = rh.ref()
        src = open(os.path.join(rh.REF_SRC, 'rayoptics', 'raytr', 'trace.py')).read()
        fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == 'iterate_ray'][0]
        opm = load_model(name)
        sm, osp = opm.seq_model, opm.optical_spec
        paths = {}

        def ref_trace(seq_model, pt0, dir0, wvl, **kw):
            if wvl not in paths:
                paths[wvl] = rh.ref_path(sm, wvl)
            kw.setdefault('first_surf', 1)
            kw.setdefault('last_surf', sm.get_num_surfaces() - 2)
            return R.raytrace.trace_raw(iter(paths[wvl]), np.array(pt0, dtype=float),
                                        np.array(dir0, dtype=float), wvl, **kw)

        class Osp:
            def __getitem__(self, k):
                return {'fov': osp.field_of_view}[k]

            def obj_coords(self, fld):
                return osp.obj_coords(fld)

        class Opm:
            def __getitem__(self, k):
                return {'seq_model': sm, 'optical_spec': Osp(),
                        'analysis_results': opm.analysis_results}[k]

        ns = dict(np=np, rt=type('rt', (), {'trace': staticmethod(ref_trace)}),
                  normalize=R.misc_math.normalize, RayPkg=TR.RayPkg, RayResult=TR.RayResult,
                  TraceError=R.traceerror.TraceError, newton=newton, fsolve=fsolve,
                  warnings=warnings, logger=logging.getLogger('ref'), mc=type('mc', (), {'p': 0}))
        exec(ast.get_source_segment(src, fn), ns)
        fld = osp.field_of_view.fields[fi]
        want, _ = ns['iterate_ray'](Opm(), sm.stop_surface, np.array([0., 0.]), fld, sm.central_wavelength())
        return want

    for name, fi in (('triplet', 1), ('thin_triplet', 1), ('exotic', 2)):
        opm = load_model(name)
        sm, osp = opm.seq_model, opm.optical_spec
        fld = osp.field_of_view.fields[fi]
        wvl = sm.central_wavelength()
        want = ref(lambda: reference_iterate_ray(name, fi))

        def our_trace(seq_model, pt0, dir0, wvl, **kw):       # engine stand-in: the oracle
            r = oracle_bundle_tracer(opm, None, np.array(pt0, dtype=float).reshape(3, 1),
                                     np.array(dir0, dtype=float).reshape(3, 1),
                                     np.array([sm.index_for_wavelength(wvl)], dtype=np.int32),
                                     dict(first_surf=1, last_surf=sm.get_num_surfaces() - 2))
            from rayoptics_b200 import raytrace as RT
            pkg, err = RT.package_ray(list(sm.path(wvl)), r['full'][:, :, 0], float(r['op'][0]),
                                      int(r['status'][0]), int(r['fail_surf'][0]),
                                      int(r['n_seg'][0]), wvl)
            if err is not None:
                raise err
            return pkg

        got = V.iterate_ray(opm, sm.stop_surface, np.array([0., 0.]), fld, wvl, trace_fn=our_trace)
        assert np.array_equal(got, want), (name, got, want)


@pytest.mark.parametrize('name,fi,wvl', [('dblgauss', 2, 486.1), ('rc', 3, 550.0), ('thin_triplet', 1, 587.6)])
def test_drivers_against_the_references_drivers(name, fi, wvl, ref):
    """trace_fan / trace_grid / trace_base / setup_pupil_coords of rayoptics_b200.trace (oracle-fed)
    against the REFERENCE's own functions of the same names (rayoptics.raytr.trace is importable)
    running on a hybrid model with the reference's trace_raw (oracle/ref_model.py).  The reference
    re-aims the field's chief ray and keeps the aim point on the field; each call here starts from
    the aim point the reference's call of the same name left."""
    opm = load_model(name)
    if wvl not in opm.seq_model.wvlns:
        wvl = opm.seq_model.central_wavelength()
    fld = opm.optical_spec.field_of_view.fields[fi]
    fan_def = lambda: [np.array([0., -1.]), np.array([0., 1.]), 11]      # noqa: E731
    grid_def = lambda: [np.array([-1., -1.]), np.array([1., 1.]), 7]     # noqa: E731
    pupils = ([0.3, -0.2], [0., 1.4])

    def cb(store):
        def f(p, pkg):
            store.append(pkg)
            return np.array([p[0], p[1], np.nan if pkg is None else pkg[1]])
        return f

    def reference_side():
        import importlib
        from oracle import ref_model
        RT, RA = ref_model.modules()
        a = load_model(name)
        H = ref_model.HybridModel(a)
        fa = a.optical_spec.field_of_view.fields[fi]
        aims = []                               # fa.aim_info after each stage

        def aim():
            aims.append(None if fa.aim_info is None else np.array(fa.aim_info, dtype=float))
        # chief ray + reference sphere
        rs_ref, cr_ref = RT.setup_pupil_coords(H, fa, wvl, 0.0)
        aim()
        # fan with an OPD callback evaluated by the reference's waveabr
        WR = importlib.import_module('rayoptics.raytr.waveabr')
        fod = a.optical_spec.fod
        f_ref = RT.trace_fan(H, fan_def(), fa, wvl, 0.0,
                             img_filter=lambda p, pkg: WR.wave_abr_full_calc(fod, fa, wvl, 0.0, pkg, cr_ref, rs_ref))
        aim()
        # grid with a callback (the reference's own np.array(grid) cannot hold raw packages under
        # numpy >= 1.24); blocked rays reach the callback as None
        seen = []
        g_ref = RT.trace_grid(H, grid_def(), fa, wvl, 0.0, form='grid', img_filter=cb(seen))
        aim()
        singles = []
        for pupil in pupils:
            try:
                singles.append(pkg_digest(RT.trace_base(H, np.array(pupil), fa, wvl, check_apertures=True)))
            except R_TraceError() as e:
                singles.append((type(e).__name__, e.surf))
            aim()
        return {'aims': aims, 'cr_pkg': pkg_digest(cr_ref[0]), 'cr': list(cr_ref[1][:3]), 'rs': list(rs_ref[:3]),
                'fan': f_ref, 'grid': g_ref, 'seen': [None if p is None else pkg_digest(p) for p in seen],
                'singles': singles}
    want = ref(reference_side)
    aims = iter(want['aims'])

    # chief ray + reference sphere
    fld.aim_info = next(aims)
    rs_own, cr_own = TR.setup_pupil_coords(opm, fld, wvl, 0.0, tracer=oracle_tracer)
    assert pkg_digest(cr_own[0]) == want['cr_pkg']
    assert np.array_equal(rs_own[0], want['rs'][0]) and np.array_equal(rs_own[1], want['rs'][1])
    assert rs_own[2] == want['rs'][2]
    for a, b in zip(cr_own[1][:3], want['cr']):
        assert np.array_equal(a, b)
    # fan with an OPD callback evaluated by this package's waveabr
    fod = opm.optical_spec.fod

    def opd_own(p, pkg):
        return W.wave_abr_full_calc(fod, fld, wvl, 0.0, pkg, cr_own, rs_own)

    fld.aim_info = next(aims)
    f_own = TR.trace_fan(opm, fan_def(), fld, wvl, 0.0, img_filter=opd_own, tracer=oracle_tracer)
    assert len(want['fan']) == len(f_own) > 3
    for (pa, va), (pb, vb) in zip(f_own, want['fan']):
        assert np.array_equal(pa, pb) and va == vb
    seen_own = []
    fld.aim_info = next(aims)
    g_own = TR.trace_grid(opm, grid_def(), fld, wvl, 0.0, form='grid', img_filter=cb(seen_own),
                          tracer=oracle_tracer)
    g_ref = want['grid']
    assert g_ref.shape == g_own.shape == (7, 7, 3) and np.array_equal(g_ref, g_own, equal_nan=True)
    assert 0 < np.isnan(g_ref[:, :, 2]).sum() < 49
    assert [None if p is None else pkg_digest(p) for p in seen_own] == want['seen']
    # single ray, error packaging
    for pupil, w in zip(pupils, want['singles']):
        fld.aim_info = next(aims)
        if isinstance(w, tuple):                # the reference raised (error class name, surface)
            with pytest.raises(type(TR.trace_pupil_rays(opm, [pupil], fld, wvl, None, 'full',
                                                        tracer=oracle_tracer,
                                                        check_apertures=True)[0].err)) as info:
                TR.trace_base(opm, np.array(pupil), fld, wvl, tracer=oracle_tracer, check_apertures=True)
            assert (type(info.value).__name__, info.value.surf) == w
        else:
            assert pkg_digest(TR.trace_base(opm, np.array(pupil), fld, wvl, tracer=oracle_tracer,
                                            check_apertures=True)) == w


def oracle_ray_fn(opm):
    from oracle import rt_oracle
    descs, n_by_wvl, wvls = T.describe_model(opm.seq_model)

    def fn(p0, d0, wvl, check_apertures=False, pt_inside_fuzz=None):
        w = np.full(p0.shape[1], opm.seq_model.index_for_wavelength(wvl), dtype=np.int32)
        return rt_oracle.trace_bundle(descs, n_by_wvl, p0, d0, w,
                                      _abi.make_opts(first_surf=1, last_surf=len(descs) - 2,
                                                     check_apertures=check_apertures,
                                                     pt_inside_fuzz=pt_inside_fuzz),
                                      want_full=True, wvls=wvls)
    return fn


@pytest.mark.parametrize('name', ['dblgauss', 'triplet', 'evenasph', 'rc'])
def test_set_vig_batched_equals_set_vig(name):
    """vigcalc.set_vig_batched (all searches in lock step, bundles) gives the vignetting
    factors of the sequential set_vig bit for bit, in far fewer launches."""
    from rayoptics_b200 import vigcalc as V
    a, b = load_model(name), load_model(name)
    for m in (a, b):
        for f in m.optical_spec.field_of_view.fields:
            f.vux = f.vlx = f.vuy = f.vly = 0.0
    V.set_vig(a, tracer=oracle_tracer)
    launches = V.set_vig_batched(b, oracle_ray_fn(b))
    fa, fb = a.optical_spec.field_of_view.fields, b.optical_spec.field_of_view.fields
    for x, y in zip(fa, fb):
        assert (x.vux, x.vlx, x.vuy, x.vly) == (y.vux, y.vlx, y.vuy, y.vly)
    assert launches < 12*len(fa) + 40


def R_TraceError():
    from oracle import ref_harness as rh
    return rh.ref().traceerror.TraceError


@pytest.mark.parametrize('name', ['dblgauss', 'triplet'])
def test_set_vig_and_apertures_equal_the_references(name, ref):
    """vigcalc.set_clear_apertures_batched and vigcalc.set_vig against the reference's
    rayoptics.raytr.vigcalc run unmodified on the hybrid model (reference trace_raw, scipy
    newton): apertures and vignetting factors bit for bit.  The reference's re-aiming is
    bypassed as in make_golden_analyses.py (placeholder chief_ray)."""
    from rayoptics_b200 import vigcalc as V

    def reference_side():
        import importlib
        from oracle import ref_model
        ref_model.modules()
        RV = importlib.import_module('rayoptics.raytr.vigcalc')
        a = load_model(name)
        H = ref_model.HybridModel(a)
        for f in a.optical_spec.field_of_view.fields:
            f.chief_ray = ((None, None, -1.0), None)
        RV.set_clear_apertures(H)
        ap = [ifc.max_aperture for ifc in H.seq_model.ifcs]
        for f in a.optical_spec.field_of_view.fields:     # vignetting from those apertures, from zero
            f.vux = f.vlx = f.vuy = f.vly = 0.0
            f.chief_ray = ((None, None, -1.0), None)
        RV.set_vig(H)
        return ap, [(f.vux, f.vlx, f.vuy, f.vly) for f in a.optical_spec.field_of_view.fields]
    ref_ap, ref_vig = ref(reference_side)
    b = load_model(name)
    V.set_clear_apertures_batched(b, oracle_bundle_fn(b))
    own_ap = [ifc.max_aperture for ifc in b.seq_model.ifcs]
    assert ref_ap[1:] == own_ap[1:]
    # vignetting from those apertures (both sides start from zero vignetting)
    for f in b.optical_spec.field_of_view.fields:
        f.vux = f.vlx = f.vuy = f.vly = 0.0
    V.set_vig(b, tracer=oracle_tracer)
    assert ref_vig == [(f.vux, f.vlx, f.vuy, f.vly) for f in b.optical_spec.field_of_view.fields]


def test_sequential_model_methods_equal_the_references(ref):
    """SequentialModel.trace_fan / trace_grid / trace_wavefront (seq/sequential.py:1006-1119): the
    reference's METHOD TEXT (the module cannot be imported: opticalglass) executed on the hybrid
    model with the reference's trace functions, against the mirror's methods (oracle-fed)."""
    def y_abr(p, xy, ray_pkg, fld, wvl, foc):
        return ray_pkg[0][-1][0][xy] - fld.ref_sphere[0][xy]

    def ht(p, wi, ray_pkg, fld, wvl, foc):
        return None if ray_pkg is None else np.array([p[0], p[1], ray_pkg[0][-1][0][1]])

    def reference_side():
        import ast
        import importlib
        from oracle import ref_model, ref_harness as rh
        RT, RA = ref_model.modules()
        src = open(os.path.join(rh.REF_SRC, 'rayoptics', 'seq', 'sequential.py')).read()
        cls = [n for n in ast.parse(src).body if isinstance(n, ast.ClassDef) and n.name == 'SequentialModel'][0]
        ns = dict(np=np, trace=RT, waveabr=importlib.import_module('rayoptics.raytr.waveabr'))
        for fn in cls.body:
            if isinstance(fn, ast.FunctionDef) and fn.name in ('trace_fan', 'trace_grid', 'trace_wavefront'):
                exec(ast.get_source_segment(src, fn), ns)
        a = load_model('dblgauss')
        H = ref_model.HybridModel(a)
        H.seq_model.opt_model = H
        for f in a.optical_spec.field_of_view.fields:          # no re-aiming by the reference
            f.chief_ray = ((None, None, -1.0), None)
        fan = ns['trace_fan'](H.seq_model, y_abr, 2, 1, num_rays=9)
        grid, _ = ns['trace_grid'](H.seq_model, ht, 1, num_rays=6, form='list', append_if_none=False)
        wf = ns['trace_wavefront'](H.seq_model, a.optical_spec.field_of_view.fields[1], 587.6, 0.0, num_rays=8)
        return fan[:3], [np.array(list(w), dtype=float) for w in grid], wf
    want_fan, want_grid, want_wf = ref(reference_side)
    b = load_model('dblgauss')
    got = b.seq_model.trace_fan(y_abr, 2, 1, num_rays=9, tracer=oracle_tracer)
    assert np.array_equal(want_fan[0], got[0]) and np.array_equal(want_fan[1], got[1]) and want_fan[2] == got[2]
    got, _ = b.seq_model.trace_grid(ht, 1, num_rays=6, form='list', append_if_none=False,
                                    tracer=oracle_tracer)
    assert len(want_grid) == len(got) == 3
    for w, g in zip(want_grid, got):
        assert np.array_equal(w, np.array(list(g), dtype=float))
    got = b.seq_model.trace_wavefront(b.optical_spec.field_of_view.fields[1], 587.6, 0.0, num_rays=8,
                                      tracer=oracle_tracer)
    assert np.array_equal(want_wf, got)


def test_find_real_enp_is_the_references(ref):
    """rayoptics_b200/wideangle.py (the wide-angle entrance pupil search) against the reference's
    raytr/wideangle.py find_real_enp run unmodified on the hybrid model: same z_enp, bit for bit,
    for every field of the fisheye fixture -- from scratch (no aim info) and with the stored value.
    The reference searches with its own trace_raw, this package's search with the oracle."""
    import warnings
    from rayoptics_b200 import wideangle as W
    b = load_model('fisheye')
    wvl = b.seq_model.central_wavelength()
    stored = [f.aim_info for f in b.optical_spec.field_of_view.fields]
    starts = [(None, s) for s in stored]

    def reference_side():
        import importlib
        from oracle import ref_model, ref_harness as rh
        ref_model.modules()
        RW = importlib.import_module('rayoptics.raytr.wideangle')
        a = load_model('fisheye')
        H = ref_model.HybridModel(a)
        out = []
        for fa, pair in zip(a.optical_spec.field_of_view.fields, starts):
            for start in pair:
                fa.aim_info = start
                with warnings.catch_warnings():
                    warnings.simplefilter('ignore')
                    z_ref, rr = RW.find_real_enp(H, a.seq_model.stop_surface, fa, wvl)
                out.append((z_ref, rr.err is None, len(rr.pkg.ray), rr.pkg.ray[-1][0], rr.pkg.op))
        fa = a.optical_spec.field_of_view.fields[1]
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            cw, rw, _ = RW.find_z_enp(H, a.seq_model.stop_surface, a.optical_spec.fod.enp_dist, fa, wvl)
        return out, cw
    want, cw = ref(reference_side)
    tf = oracle_trace_fn(b)
    k = 0
    for fb, pair in zip(b.optical_spec.field_of_view.fields, starts):
        for start in pair:
            fb.aim_info = start
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                z_own, rr_own = W.find_real_enp(b, b.seq_model.stop_surface, fb, wvl, trace_fn=tf)
            z_ref, ok, n_ray, p_last, op = want[k]
            k += 1
            assert z_own == z_ref
            assert abs(z_ref - pair[1]) < 1e-9
            # the second return value is the reference's: RayResult of the last ray traced
            assert (rr_own.err is None) == ok and len(rr_own.pkg.ray) == n_ray
            assert np.array_equal(rr_own.pkg.ray[-1][0], p_last) and rr_own.pkg.op == op
    assert k == len(want)
    # the older secant-only search from the paraxial pupil, and the pupil curve across the field
    fb = b.optical_spec.field_of_view.fields[1]
    fod = b.optical_spec.fod
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        cg, rg, res = W.find_z_enp(b, b.seq_model.stop_surface, fod.enp_dist, fb, wvl, trace_fn=tf)
    assert np.array_equal(cw, cg) and res.converged and abs(cg[2] - stored[1]) < 1e-5
    rel = b.optical_spec.field_of_view.is_relative
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        flds, angs, hts, zs = W.eval_z_enp_curve(b, printout=False, trace_fn=tf, num_fields=5)
    assert b.optical_spec.field_of_view.is_relative == rel and len(flds) == 5
    assert angs[0] == 0.0 and abs(angs[-1] - b.optical_spec.field_of_view.value) < 1e-9
    assert zs[0] == fod.enp_dist and all(z1 < z0 for z0, z1 in zip(zs, zs[1:]))   # the pupil walks towards the lens
    assert abs(zs[-1] - stored[-1]) < 1e-9 and hts[0] == 0.0


def _hybrid_with_powers(opm):
    """the reference's analysis layer on the mirror model, with what its Coddington trace reads
    from a SequentialModel: ``rndx`` and the interfaces' ``delta_n`` (seq/sequential.py:628-657,
    recomputed here from the index table, not taken from model.Surface.delta_n)"""
    from oracle import ref_model
    H = ref_model.HybridModel(opm)
    sm = opm.seq_model
    H.seq_model.rndx = sm.rndx
    ref = sm.index_for_wavelength(sm.central_wavelength())
    n_before = sm.rndx[0][ref]
    for i, ifc in enumerate(H.seq_model.ifcs[:len(sm.gaps)]):
        n_after = sm.rndx[i][ref]*(1 if sm.z_dir[i] > 0 else -1)
        ifc.delta_n = n_after - n_before
        n_before = n_after
        if hasattr(sm.ifcs[i], 'profile'):
            assert sm.ifcs[i].delta_n == ifc.delta_n
            assert sm.ifcs[i].optical_power == ifc.optical_power
    return H


@pytest.mark.parametrize('name', ['dblgauss', 'triplet', 'rc', 'evenasph', 'cellphone', 'telecentric'])
def test_trace_module_call_surface_equals_the_references(name, capsys, ref):
    """refocus, trace_with_opd, trace_astigmatism(_curve), the Coddington trace, the DataFrame
    listings and the printers of rayoptics.raytr.trace, run by the reference on the hybrid model
    and here on the batched drivers (oracle in the tracer seam): identical numbers / text."""
    import contextlib
    import io
    from rayoptics_b200.model import Field
    P1, V1 = np.array([0., 1., 0.]), np.array([0., -0.1, 1.])/np.linalg.norm([0., -0.1, 1.])
    P2, V2 = np.array([0., -1., 0.]), np.array([0., 0.1, 1.])/np.linalg.norm([0., 0.1, 1.])
    spherical = name in ('dblgauss', 'triplet', 'telecentric')
    opd_pupils = ([0., 0.6], [0.4, -0.3])

    def df_values(df):
        return list(df.index), list(df.columns), digest([[np.asarray(x) for x in df[col]] for col in df.columns])

    def reference_side():
        from oracle import ref_model
        RT, RA = ref_model.modules()
        a = load_model(name)
        H = _hybrid_with_powers(a)
        fa = a.optical_spec.field_of_view.fields[-1]
        wvl = a.seq_model.central_wavelength()
        out = {'refocus': RT.refocus(H),
               'astigmatism': [RT.trace_astigmatism(H, fa, wvl, foc) for foc in (0.0, 0.02)]}
        # trace_astigmatism_curve: the reference's loop body (trace.py:812-822) on the reference's
        # functions (its own Field class needs opticalglass to import, the mirror's Field stands in)
        fov = a.optical_spec.field_of_view
        fld = Field(fov=fov)
        sw, tw = [], []
        for f in np.linspace(0., fov.max_field()[0], num=5):
            fld.yv = f
            ref_sphere, cr_pkg = RT.setup_pupil_coords(H, fld, wvl, 0.0)
            fld.chief_ray, fld.ref_sphere = cr_pkg, ref_sphere
            s_foc, t_foc = RT.trace_astigmatism(H, fld, wvl, 0.0)
            sw.append(s_foc)
            tw.append(t_foc)
        out['curve'] = (sw, tw)
        # Coddington trace along the chief ray of the outer field
        pw = RT.trace_ray(H, [0., 0.], fa, wvl)[0]
        out['chief'] = {'n_seg': len(pw.ray), 'op': pw.op,
                        'ray': digest(np.array([np.concatenate([s.p, s.d, [s.dst], s.nrml]) for s in pw.ray]))}
        if spherical:
            out['coddington'] = [RT.trace_coddington_fan(H, pw, foc=foc) for foc in (None, 0.01)]
            out['coddington_astigmatism'] = RT.trace_astigmatism_coddington_fan(H, fa, wvl, 0.0)
        # OPD of single rays (chief ray present on the field: no re-aiming)
        out['opd'] = []
        for pupil in opd_pupils:
            fa.chief_ray = ((None, None, -1.0), None)
            rw = RT.trace_with_opd(H, list(pupil), fa, wvl, 0.01)
            out['opd'].append((rw[1], rw[2], rw[3], rw[0][-1][0]))
        out['all_fields'] = df_values(RT.trace_all_fields(H))
        out['ray_pkg_index'] = RT.ray_pkg(pw).index.tolist()
        # printers
        text = io.StringIO()
        with contextlib.redirect_stdout(text):
            RT.list_ray(pw)
            RT.list_ray((pw, None), tfrms=[(np.identity(3), np.array([0., 0., float(k)])) for k in range(len(pw.ray))],
                        start=2)
            RT.list_in_out_dir(list(H.seq_model.path(wvl)), pw.ray)
        out['printed'] = text.getvalue()
        out['intersect'] = RT.intersect_2_lines(P1, V1, P2, V2)
        return out
    want = ref(reference_side)

    b = load_model(name)
    kw = dict(tracer=oracle_tracer)
    fb = b.optical_spec.field_of_view.fields[-1]
    wvl = b.seq_model.central_wavelength()

    assert want['refocus'] == TR.refocus(b, **kw)

    for w, foc in zip(want['astigmatism'], (0.0, 0.02)):
        got = TR.trace_astigmatism(b, fb, wvl, foc, **kw)
        assert w == got and np.isfinite(got).all()
    fov = b.optical_spec.field_of_view
    fg, sg, tg = TR.trace_astigmatism_curve(b, num_points=5, **kw)
    sw, tw = want['curve']
    assert list(fg) == list(np.linspace(0., fov.max_field()[0], num=5)) and sw == sg and tw == tg
    assert fov.max_field()[0] > 0 and abs(sg[0] - tg[0]) < 1e-9 < abs(sg[-1] - tg[-1])

    # Coddington trace along the chief ray of the outer field
    pg = TR.trace_ray(b, [0., 0.], fb, wvl, **kw)[0]
    assert_pkg_equals(pg, want['chief'])
    if spherical:                               # spherical surfaces only
        for w, foc in zip(want['coddington'], (None, 0.01)):
            got = TR.trace_coddington_fan(b, pg, foc=foc)
            assert w == got and np.isfinite(got).all()
        assert want['coddington_astigmatism'] == TR.trace_astigmatism_coddington_fan(b, fb, wvl, 0.0, **kw)

    # OPD of single rays (chief ray present on the field: no re-aiming)
    for pupil, w in zip(opd_pupils, want['opd']):
        fb.chief_ray = ((None, None, -1.0), None)
        rg = TR.trace_with_opd(b, list(pupil), fb, wvl, 0.01, **kw)
        assert w[0] == rg[1] and w[1] == rg[2] and w[2] == rg[3]
        assert np.array_equal(w[3], rg[0][-1][0])

    # DataFrames
    assert df_values(TR.trace_all_fields(b, **kw)) == want['all_fields']
    assert TR.ray_pkg(pg).index.tolist() == want['ray_pkg_index']

    # printers
    capsys.readouterr()
    TR.list_ray(pg)
    TR.list_ray((pg, None), tfrms=[(np.identity(3), np.array([0., 0., float(k)])) for k in range(len(pg.ray))], start=2)
    TR.list_in_out_dir(list(b.seq_model.path(wvl)), pg.ray)
    got = capsys.readouterr().out
    assert want['printed'] == got and len(got.splitlines()) > 2*len(pg.ray)

    assert want['intersect'] == TR.intersect_2_lines(P1, V1, P2, V2)


@pytest.mark.parametrize('name,use_parax', [('dblgauss', False), ('dblgauss', True), ('triplet', False),
                                            ('relay_fno', False)])
def test_set_pupil_and_bisection_equal_the_references(name, use_parax, capsys, ref):
    """vigcalc.set_pupil (stop size -> pupil specification + vignetting), set_stop_aperture and
    calc_vignetted_ray_by_bisection against rayoptics.raytr.vigcalc on the hybrid model."""
    import contextlib
    import io
    from rayoptics_b200 import vigcalc as V
    starts = ((1, [0., 1.]), (0, [-1., 0.]))

    def reference_side():
        import importlib
        from oracle import ref_model
        ref_model.modules()
        RV = importlib.import_module('rayoptics.raytr.vigcalc')
        a = load_model(name)
        H = ref_model.HybridModel(a)
        H.update_model = a.update_model

        def keep():
            for f in a.optical_spec.field_of_view.fields:
                f.chief_ray = ((None, None, -1.0), None)
        # bisection search of the upper y pupil edge of the outer field
        fa = a.optical_spec.field_of_view.fields[-1]
        wvl = a.seq_model.central_wavelength()
        bisection = []
        for xy, start in starts:
            keep()
            vw, cw, pw = RV.calc_vignetted_ray_by_bisection(H, xy, np.array(start), fa, wvl)
            bisection.append((vw, cw, len(pw[0])))
        # a smaller stop: the pupil specification follows
        stop = a.seq_model.stop_surface
        r = 0.9*a.seq_model.ifcs[stop].max_aperture
        H.seq_model.ifcs[stop].set_max_aperture(r)
        a.seq_model.ifcs[stop].set_max_aperture(r)
        keep()
        a_update = a.update_model

        def update_and_keep(**k):
            a_update(**k)
            keep()
        H.update_model = update_and_keep
        text = io.StringIO()
        with contextlib.redirect_stdout(text):
            RV.set_pupil(H, use_parax=use_parax)
        return {'bisection': bisection, 'pupil': a.optical_spec.pupil.value,
                'axial_limited': text.getvalue().count('Axial bundle limited'),
                'vig': [(f.vux, f.vlx, f.vuy, f.vly) for f in a.optical_spec.field_of_view.fields]}
    want = ref(reference_side)
    capsys.readouterr()
    b = load_model(name)
    kw = dict(tracer=oracle_tracer)
    fb = b.optical_spec.field_of_view.fields[-1]
    wvl = b.seq_model.central_wavelength()
    for (xy, start), (vw, cw, n_pw) in zip(starts, want['bisection']):
        vg, cg, pg = V.calc_vignetted_ray_by_bisection(b, xy, np.array(start), fb, wvl, **kw)
        assert vw == vg and cw == cg and n_pw == len(pg[0])
    # a smaller stop: the pupil specification follows
    stop = b.seq_model.stop_surface
    r = 0.9*b.seq_model.ifcs[stop].max_aperture
    b.seq_model.ifcs[stop].set_max_aperture(r)
    before = b.optical_spec.pupil.value
    V.set_pupil(b, use_parax=use_parax, **kw)
    assert want['pupil'] == b.optical_spec.pupil.value != before
    # (the reference's image-space f/# comes out negative for the relay: kept, it is its number)
    assert abs(abs(b.optical_spec.pupil.value/before) - (1/0.9 if b.optical_spec.pupil.key[1] == 'f/#' else 0.9)) < 0.02
    assert want['vig'] == [(y.vux, y.vlx, y.vuy, y.vly) for y in b.optical_spec.field_of_view.fields]
    assert capsys.readouterr().out.count('Axial bundle limited') == want['axial_limited']


def oracle_trace_fn(opm):
    """trace_fn= seam (one ray, the drop-in ``raytrace.trace`` signature) fed by the oracle"""
    from rayoptics_b200 import raytrace as RT
    sm = opm.seq_model

    def fn(seq_model, pt0, dir0, wvl, **kw):
        opts = dict(first_surf=1, last_surf=sm.get_num_surfaces() - 2)
        opts.update({k: v for k, v in kw.items() if k in TR._TRACE_RAW_KEYS})
        r = oracle_bundle_tracer(opm, None, np.array(pt0, dtype=float).reshape(3, 1),
                                 np.array(dir0, dtype=float).reshape(3, 1),
                                 np.array([sm.index_for_wavelength(wvl)], dtype=np.int32), opts)
        pkg, err = RT.package_ray(list(sm.path(wvl)), r['full'][:, :, 0], float(r['op'][0]),
                                  int(r['status'][0]), int(r['fail_surf'][0]), int(r['n_seg'][0]), wvl)
        if err is not None:
            raise err
        return pkg
    return fn


def test_aperture_lists_and_stop_aperture():
    """set_clear_apertures with include / avoid lists (vigcalc.py:45-80) in both forms, and
    set_stop_aperture (vigcalc.py:104-115): the stop takes the height of the unvignetted axial
    marginal ray, everything else is left alone, the vignetting is recomputed."""
    from rayoptics_b200 import vigcalc as V
    a, b, c = load_model('dblgauss'), load_model('dblgauss'), load_model('dblgauss')
    n = a.seq_model.get_num_surfaces()
    stop = a.seq_model.stop_surface
    orig = [ifc.max_aperture for ifc in a.seq_model.ifcs]
    for m in (a, b, c):
        for ifc in m.seq_model.ifcs:
            ifc.set_max_aperture(1.25*ifc.max_aperture)
    big = [ifc.max_aperture for ifc in a.seq_model.ifcs]
    V.set_clear_apertures(a, oracle_trace_fn(a), include_list=[2, 3, stop])
    V.set_clear_apertures_batched(b, oracle_bundle_fn(b), avoid_list=[i for i in range(n) if i not in (2, 3, stop)])
    for i in range(n):
        ap_a, ap_b = a.seq_model.ifcs[i].max_aperture, b.seq_model.ifcs[i].max_aperture
        assert ap_a == ap_b
        assert (ap_a != big[i]) == (i in (2, 3, stop))
    rayset = V.trace_boundary_rays(c, oracle_trace_fn(c))
    assert V.max_aperture_at_surf([rayset[0]], stop) == a.seq_model.ifcs[stop].max_aperture
    assert V.max_aperture_at_surf(rayset, n + 3) is None
    # set_stop_aperture: axial vignetting cleared, stop := axial marginal ray height, set_vig
    f0 = c.optical_spec.field_of_view.fields[0]
    f0.vuy = f0.vly = 0.2
    V.set_stop_aperture(c, trace_fn=oracle_trace_fn(c), tracer=oracle_tracer)
    ray = TR.trace_base(c, np.array([0., 1.]), f0, c.seq_model.central_wavelength(),
                        apply_vignetting=False, tracer=oracle_tracer)
    assert abs(c.seq_model.ifcs[stop].max_aperture - abs(ray[0][stop][0][1])) < 1e-9
    assert [ifc.max_aperture for i, ifc in enumerate(c.seq_model.ifcs) if i != stop] == \
           [x for i, x in enumerate(big) if i != stop]
    assert abs(f0.vuy) < 1e-5 and abs(f0.vly) < 1e-5          # the stop is the limiting aperture on axis
    assert orig[stop] > 0


@pytest.mark.parametrize('name,fi', [('dblgauss', 2), ('triplet', 1), ('evenasph', 1)])
def test_iterate_ray_raw_equals_the_references(name, fi, ref):
    """vigcalc.iterate_ray_raw against rayoptics.raytr.trace.iterate_ray_raw (imported, run on
    the reference's own trace_raw over reference surfaces): same aim point, 1-D (newton) and
    2-D (fsolve) branches."""
    from rayoptics_b200 import vigcalc as V
    opm = load_model(name)
    sm, osp = opm.seq_model, opm.optical_spec
    fod = osp.fod
    wvl = sm.central_wavelength()
    fld = osp.field_of_view.fields[fi]
    pt0, d0 = osp.obj_coords(fld)
    one = oracle_trace_fn(opm)
    args = (fod.obj_dist + fod.enp_dist, fod.enp_radius, wvl, True)
    cases = ((np.array([0., 0.]), pt0), (np.array([0.05, -0.02]), pt0),
             (np.array([0., 0.1]), pt0 + np.array([0.3, 0., 0.])))

    def reference_side():
        from oracle import ref_model, ref_harness as rh
        RT, RA = ref_model.modules()
        out = []
        for target, p0 in cases:
            want, rr_w = RT.iterate_ray_raw(rh.ref_path(sm, wvl), sm.stop_surface, target, p0, d0, *args)
            out.append((want, rr_w.pkg.ray[-1][0]))
        return out
    for (target, p0), (want, p_last) in zip(cases, ref(reference_side)):
        got, rr_g = V.iterate_ray_raw(sm.path(wvl), sm.stop_surface, target, p0, d0, *args,
                                      trace_raw_fn=lambda path, p, d, w: one(sm, p, d, w))
        assert np.array_equal(want, got), (name, target)
        assert rr_g[1] is None and np.array_equal(p_last, rr_g[0][0][-1][0])
    got, rr = V.iterate_ray_raw(sm.path(wvl), None, np.array([0.1, 0.2]), pt0, d0, *args)
    assert np.array_equal(got, [0.1, 0.2]) and rr is None


@pytest.mark.parametrize('name', ['dblgauss', 'triplet', 'rc', 'cellphone'])
def test_paraxial_vignetting_equals_the_references(name, ref):
    """vigcalc.paraxial_vignetting / apply_paraxial_vignetting against the reference's METHOD TEXT
    (parax/paraxialdesign.py:1023-1050 -- the module needs opticalglass to import) and
    rayoptics.raytr.trace.apply_paraxial_vignetting run on shims of the same paraxial data."""
    from rayoptics_b200 import vigcalc as V
    rels = (0.0, 0.5, 1.0)

    def tighter(m):                                    # tighter apertures so that something vignettes
        for ifc in m.seq_model.ifcs[1:-1]:
            ifc.set_max_aperture(0.8*ifc.max_aperture)
        return m

    def reference_side():
        import ast
        from oracle import ref_model, ref_harness as rh
        RT, RA = ref_model.modules()
        src = open(os.path.join(rh.REF_SRC, 'rayoptics', 'parax', 'paraxialdesign.py')).read()
        cls = [n for n in ast.parse(src).body if isinstance(n, ast.ClassDef) and n.name == 'ParaxialModel'][0]
        fn = [f for f in cls.body if isinstance(f, ast.FunctionDef) and f.name == 'paraxial_vignetting'][0]
        ns = dict(mc=type('mc', (), {'ht': 0, 'slp': 1}))
        exec(ast.get_source_segment(src, fn), ns)
        a = tighter(load_model(name))
        H = ref_model.HybridModel(a)
        for ref_ifc, ifc in zip(H.seq_model.ifcs, a.seq_model.ifcs):
            ref_ifc.set_max_aperture(ifc.max_aperture)
        fod = a.optical_spec.fod
        pm = type('PM', (), {})()
        pm.seq_model, pm.ax, pm.pr = H.seq_model, fod.ax_ray, fod.pr_ray
        pm.paraxial_vignetting = lambda rel_fov=1: ns['paraxial_vignetting'](pm, rel_fov)
        vig = [pm.paraxial_vignetting(rel) for rel in rels]
        H.parax_model = pm
        RT.apply_paraxial_vignetting(H)
        return vig, [(f.vly, f.vuy) for f in a.optical_spec.field_of_view.fields]
    want_vig, want_fields = ref(reference_side)
    b = tighter(load_model(name))
    for rel, w in zip(rels, want_vig):
        assert w == V.paraxial_vignetting(b, rel)
    TR.apply_paraxial_vignetting(b)
    got = [(f.vly, f.vuy) for f in b.optical_spec.field_of_view.fields]
    assert want_fields == got
    assert any(v != 0 for pair in got for v in pair)


def oracle_trace_raw_fn(path, pt0, dir0, wvl, **kw):
    """trace_raw_fn= seam (an explicit path list, e.g. a reverse path) fed by the oracle"""
    from oracle import rt_oracle
    from rayoptics_b200 import raytrace as RT
    segs = list(path)
    descs, ns = T.describe_path(segs)
    opts = {k: v for k, v in kw.items() if k in TR._TRACE_RAW_KEYS}
    r = rt_oracle.trace_ray(descs, ns, np.array(pt0, dtype=float), np.array(dir0, dtype=float),
                            _abi.make_opts(**opts))
    full = np.full((len(descs), 10), np.nan)
    full[:r['n_seg']] = r['ray']
    pkg, err = RT.package_ray(segs, full, r['op'], r['status'], r['fail_surf'], r['n_seg'], wvl)
    if err is not None:
        raise err
    return pkg


def _real_height_model(name):
    """a fixture re-specified by REAL image heights: ('image', 'real height') fields at the
    heights its own chief rays reach"""
    opm = load_model(name)
    osp, sm = opm.optical_spec, opm.seq_model
    sm.ifcs[0].interact_mode = 'dummy'         # as in every reference OpticalModel (sequential.py:600)
    wvl = sm.central_wavelength()
    hts = []
    for f in osp.field_of_view.fields:
        f.aim_info = None
        pkg = TR.trace_base(opm, np.array([0., 0.]), f, wvl, tracer=oracle_tracer)
        hts.append(pkg[0][-1][0][:2].copy())
    fov = osp.field_of_view
    fov.key, fov.is_relative = ('image', 'real height'), False
    for f, h in zip(fov.fields, hts):
        f.x, f.y, f.aim_info = float(h[0]), float(h[1]), None
    fov.value = max(abs(h[1]) for h in hts)
    return opm, hts


@pytest.mark.parametrize('name', ['dblgauss', 'triplet', 'relay_fno', 'cellphone'])
def test_real_image_height_fields_equal_the_references(name, ref):
    """('image', 'real height') fields (Zemax FTYP 3): wideangle.eval_real_image_ht -- the chief ray
    iterated backwards through the stop centre on SequentialModel.reverse_path -- against the
    reference's own eval_real_image_ht (its iterate_ray_raw, its trace_raw on reference surfaces in
    the reversed path); then obj_coords / ray_start_from_osp: the forward chief ray lands on the
    requested image height."""
    from rayoptics_b200 import wideangle as W

    def reference_side():
        import importlib
        from oracle import ref_model
        ref_model.modules()
        RW = importlib.import_module('rayoptics.raytr.wideangle')
        a, _ = _real_height_model(name)
        H = ref_model.HybridModel(a)
        wvl = a.seq_model.central_wavelength()
        return [RW.eval_real_image_ht(H, fa, wvl) for fa in a.optical_spec.field_of_view.fields]
    want = ref(reference_side)
    b, hts = _real_height_model(name)
    wvl = b.seq_model.central_wavelength()
    b.optical_spec._trace_raw_fn = oracle_trace_raw_fn
    assert len(want) == len(b.optical_spec.field_of_view.fields)
    for fb, h, ((pw, dw), zw) in zip(b.optical_spec.field_of_view.fields, hts, want):
        (pg, dg), zg = W.eval_real_image_ht(b, fb, wvl, trace_raw_fn=oracle_trace_raw_fn)
        assert np.array_equal(pw, pg) and np.array_equal(dw, dg) and zw == zg
        # forward: the start ray built from obj_coords (which stores the implied aim point) hits h
        if name == 'cellphone' and fb is b.optical_spec.field_of_view.fields[-1]:
            continue     # the reverse secant iteration runs away at this lens' extreme field -- in the
                         # reference too (same numbers above); nothing to check forwards
        pkg = TR.trace_base(b, np.array([0., 0.]), fb, wvl, tracer=oracle_tracer)
        assert fb.aim_info is not None
        assert np.abs(pkg[0][-1][0][:2] - h).max() < 2e-6*max(1.0, np.abs(h).max())
        stop = b.seq_model.stop_surface
        assert np.abs(pkg[0][stop][0][:2]).max() < 1e-3          # the reverse iteration stops at scipy newton's default tolerance
    # the batched start rays (one reverse iteration per FIELD, then whole grids) are the per-ray ones
    from oracle import rt_oracle
    osp, sm = b.optical_spec, b.seq_model
    flds = osp.field_of_view.fields[:-1] if name == 'cellphone' else osp.field_of_view.fields
    recs, eprad, z_pupil = osp.grid_fields(flds)
    px = np.array([-0.7, 0.0, 0.4, 1.0])
    spec = E.PupilGridSpec(recs, [0], px, px, eprad, z_pupil, apply_vignetting=True, flip_z_dir=sm.z_dir[0])
    p, d, wv, _ = rt_oracle.grid_start_rays(spec.c_spec(), 0, spec.n_rays)
    k = 0
    for fld in flds:
        for x in px:
            for y in px:
                pt0, dir0 = osp.ray_start_from_osp(fld.apply_vignetting(np.array([x, y])), fld, 'rel pupil')
                if dir0[2]*sm.z_dir[0] < 0:
                    dir0 = -dir0
                assert np.array_equal(p[:, k], pt0) and np.array_equal(d[:, k], dir0)
                k += 1


@pytest.mark.parametrize('fname', ['zemax/tests/US05831776-1.zmx', 'zemax/tests/US08427765-1.ZMX'])
def test_zemax_real_image_height_files(fname):
    """The two bundled Zemax files with FTYP 3 (fields given as real image heights): the chief ray
    of every field lands on its height and passes the stop centre."""
    import warnings
    from rayoptics_b200 import zmx, seq
    opm = zmx.open_zmx(os.path.join(lens_files(), fname), glass_map=seq.SubstituteGlasses())
    osp, sm = opm.optical_spec, opm.seq_model
    assert tuple(osp.field_of_view.key) == ('image', 'real height')
    osp._trace_raw_fn = oracle_trace_raw_fn
    wvl = sm.central_wavelength()
    for fld in osp.field_of_view.fields:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            pkg = TR.trace_base(opm, np.array([0., 0.]), fld, wvl, tracer=oracle_tracer)
        want = np.array([fld.x, fld.y])*(osp.field_of_view.value if osp.field_of_view.is_relative else 1.0)
        assert np.abs(pkg[0][-1][0][:2] - want).max() < 1e-4*max(1.0, np.abs(want).max()), (fld.y, pkg[0][-1][0])
        assert np.abs(pkg[0][sm.stop_surface][0][:2]).max() < 1e-2


def test_engine_failures_stay_loud_inside_the_searches():
    """The aiming / pupil searches absorb per-ray TraceErrors and scipy's own 'did not converge'
    the way the reference does -- but an engine failure (EngineError, a CUDA RuntimeError) raised
    by the tracer inside a residual function must come out, not turn into 'no solution'."""
    from rayoptics_b200 import vigcalc as V, wideangle as W
    opm = load_model('dblgauss')
    sm, osp = opm.seq_model, opm.optical_spec
    fld, wvl = osp.field_of_view.fields[2], sm.central_wavelength()

    def broken(*a, **k):
        raise _abi.EngineError('libb200rt error -2: simulated device failure')

    def cuda_broken(*a, **k):
        raise RuntimeError('CUDA error: an illegal memory access was encountered')
    for bad in (broken, cuda_broken):
        with pytest.raises(RuntimeError, match='simulated device failure|illegal memory'):
            V.iterate_ray(opm, sm.stop_surface, np.array([0., 0.]), fld, wvl, trace_fn=bad)
        with pytest.raises(RuntimeError, match='simulated device failure|illegal memory'):
            V.aim_chief_ray(opm, fld, wvl, bad)
        with pytest.raises(RuntimeError, match='simulated device failure|illegal memory'):
            V.trace_boundary_rays(opm, bad)
        with pytest.raises(RuntimeError, match='simulated device failure|illegal memory'):
            V.iterate_ray_raw(sm.path(wvl), sm.stop_surface, np.array([0., 0.]), *osp.obj_coords(fld),
                              1e10, 10.0, wvl, True, trace_raw_fn=bad)
    fish = load_model('fisheye')
    ff = fish.optical_spec.field_of_view.fields[2]
    ff.aim_info = None
    for bad in (broken, cuda_broken):
        with pytest.raises(RuntimeError, match='simulated device failure|illegal memory'):
            W.find_real_enp(fish, fish.seq_model.stop_surface, ff, fish.seq_model.central_wavelength(), trace_fn=bad)
    assert V.solver_gave_up(RuntimeError('Failed to converge after 50 iterations, value is 1.0.'))
    assert not V.solver_gave_up(_abi.EngineError('Failed to converge'))     # not scipy's class


def test_real_pupil_search_decisions_equal_the_references(monkeypatch, ref):
    """Every branch of the wide-angle pupil search (scan direction reversal, first-surface misses,
    single success, beam edges, no crossing) against the reference's find_real_enp: both run on the
    same SYNTHETIC 'ray' -- a scripted stop height h(z) with windows where the trace fails in
    scripted ways -- substituted for enp_z_coordinate in the two modules.  Same z_enp, same
    sequence of z values evaluated (stored as their count per scenario and one digest())."""
    import warnings
    from rayoptics_b200 import wideangle as W, raytrace as BR
    opm = load_model('fisheye')
    stop = opm.seq_model.stop_surface
    wvl = opm.seq_model.central_wavelength()
    fld = opm.optical_spec.field_of_view.fields[3]
    rng = np.random.default_rng(77)
    n_ifc = opm.seq_model.get_num_surfaces()

    def scenario():
        z0 = opm.optical_spec.fod.enp_dist
        zc = z0*rng.uniform(-0.6, 1.8)                       # where the chief ray crosses the stop centre
        slope, cubic = rng.uniform(0.05, 2.0)*rng.choice([-1, 1]), rng.uniform(0, 0.02)
        lo, hi = sorted(z0*rng.uniform(-1.5, 2.5, 2))        # window in which rays get through
        if rng.random() < 0.3:
            lo, hi = -1e9, 1e9
        if rng.random() < 0.15:                              # a sliver: single success / edges
            mid = z0*rng.uniform(0.2, 1.4)
            lo, hi = mid - abs(z0)*0.02, mid + abs(z0)*0.02
        if rng.random() < 0.25:                              # crossing just inside one end of the window
            w = abs(z0)*rng.uniform(0.1, 0.6)
            eps = abs(z0)/16*rng.uniform(0.05, 0.9)
            lo, hi = (zc - eps, zc - eps + w) if rng.random() < 0.5 else (zc + eps - w, zc + eps)
        kind_lo, kind_hi = rng.integers(0, 3, 2)             # 0: miss at 1, 1: miss later, 2: blocked
        return dict(h=lambda z: slope*(z - zc) + cubic*(z - zc)**3, lo=lo, hi=hi, kinds=(kind_lo, kind_hi))

    def synthetic(sc, errs, RayPkg, RayResult, log):
        def fn(z_enp, *args):
            log.append(float(z_enp))
            ray = [[np.zeros(3), np.array([0., 0., 1.]), 0.0, np.array([0., 0., 1.])] for _ in range(n_ifc)]
            if sc['lo'] < z_enp < sc['hi']:
                ray[stop][0] = np.array([0., sc['h'](z_enp), 0.])
                return ray[stop][0], RayResult(RayPkg(ray, 0.0, wvl), None)
            kind = sc['kinds'][0 if z_enp <= sc['lo'] else 1]
            if kind == 2:
                err = errs.TraceRayBlockedError(None, np.zeros(3))
                err.surf = 2
            else:
                err = errs.TraceMissedSurfaceError(None, None)
                err.surf = 1 if kind == 0 else 3
            err.ray_pkg = (ray[:err.surf + 1], 0.0, wvl)
            return np.array([0., 0., 0.]), RayResult(RayPkg(ray[:err.surf + 1], 0.0, wvl), err)
        return fn

    scenarios = [scenario() for _ in range(1500)]

    def run(module, model, f, errs, RayPkg, RayResult):
        """per scenario: z_enp found by module.find_real_enp (or the exception's class name), and
        the z values it evaluated"""
        found, logs = [], []
        for sc in scenarios:
            log = []
            monkeypatch.setattr(module, 'enp_z_coordinate', synthetic(sc, errs, RayPkg, RayResult, log))
            f.aim_info = None
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                try:
                    z = module.find_real_enp(model, stop, f, wvl)[0]
                except Exception as e:      # noqa: BLE001 - e.g. no successful ray at all: start_z is None
                    z = type(e).__name__
            found.append(z)
            logs.append(log)
        return found, logs

    def reference_side():
        import importlib
        from oracle import ref_model, ref_harness as rh
        ref_model.modules()
        RW = importlib.import_module('rayoptics.raytr.wideangle')
        a = load_model('fisheye')
        found, logs = run(RW, ref_model.HybridModel(a), a.optical_spec.field_of_view.fields[3],
                          rh.ref().traceerror, RW.RayPkg, RW.RayResult)
        return found, [len(log) for log in logs], digest(logs)
    want, want_counts, want_logs = ref(reference_side)
    got, logs = run(W, opm, fld, BR, TR.RayPkg, TR.RayResult)
    assert [len(log) for log in logs] == want_counts and digest(logs) == want_logs
    outcomes = set()
    for trial, (sc, w, g) in enumerate(zip(scenarios, want, got)):
        assert (w == g) or (isinstance(w, float) and np.isnan(w) and np.isnan(g)), trial
        outcomes.add('error' if isinstance(w, str) else
                     'crossing' if abs(sc['h'](w)) < 1e-6 else 'no crossing')
    assert len(got) == len(want) == 1500 and outcomes == {'error', 'crossing', 'no crossing'}


@pytest.mark.parametrize('name', ['dblgauss', 'relay_na', 'fisheye'])
def test_aim_point_and_aim_direction_pupils(name, ref):
    """trace_base / trace_safe with pupil_type 'aim pt' and 'aim dir' (trace.py:253-310,
    opticalspec.py:332-336,369-371): the reference's trace_base on the hybrid model against the
    bundle path here, whole rays (the segments' p, d, dst as digest())."""
    b = load_model(name)
    wvl = b.seq_model.central_wavelength()
    fod = b.optical_spec.fod
    fb = b.optical_spec.field_of_view.fields[1]
    angular = b.optical_spec.pupil.key[1] != 'epd'
    if angular:
        ptype, pupils = 'aim dir', [np.array([0.0, 0.02]), np.array([0.01, -0.015]), np.array([-0.02, 0.0])]
    else:
        r = fod.enp_radius
        ptype, pupils = 'aim pt', [np.array([0.0, 0.3*r]), np.array([0.2*r, -0.4*r]), np.array([-0.5*r, 0.1*r])]

    def summary(pkg):
        return len(pkg[0]), pkg[1], digest([tuple(seg)[:3] for seg in pkg[0]])

    def reference_side():
        from oracle import ref_model
        RT, RA = ref_model.modules()
        a = load_model(name)
        H = ref_model.HybridModel(a)
        fa = a.optical_spec.field_of_view.fields[1]
        out = []
        for pupil in pupils:
            for check in (False, True):
                try:
                    out.append(summary(RT.trace_base(H, pupil.copy(), fa, wvl, pupil_type=ptype,
                                                     check_apertures=check)))
                except Exception as e:      # noqa: BLE001 - a reference TraceError
                    out.append(type(e).__name__)
        return out
    want = iter(ref(reference_side))
    for pupil in pupils:
        for check in (False, True):
            try:
                got = summary(TR.trace_base(b, pupil.copy(), fb, wvl, pupil_type=ptype, check_apertures=check,
                                            bundle_tracer=oracle_bundle_tracer))
            except Exception as e:      # noqa: BLE001
                got = type(e).__name__
            assert got == next(want)
    res = TR.trace_pupil_rays(b, pupils, fb, wvl, None, 'full', pupil_type=ptype,
                              bundle_tracer=oracle_bundle_tracer)
    assert len(res) == 3 and all(r.pkg is not None for r in res)


def test_post_import_update_sets_aims_and_apertures():
    """OpticalModel.update_optical_properties -- the ray-traced part of the reference's post-import
    update_model (opticalmodel.py:318-354, cmdproc.py:85-94, zmxread.py:247-249): chief rays
    aimed at the stop centre; a file without aperture data gets clear apertures from the boundary
    rays (the stop from the axial bundle), a file with some CIR records keeps those and gets the
    rest; DIAM kinds decide for .zmx files."""
    from rayoptics_b200 import seq, zmx, vigcalc as V
    sample = os.path.join(os.path.dirname(__file__), 'golden', 'samples', 'triplet_fict.seq')
    lines = open(sample).read().splitlines()
    tmp_dir = os.path.dirname(sample)
    path, part_path = os.path.join(tmp_dir, '_tmp_nocir.seq'), sample
    try:
        open(path, 'w').write(chr(10).join(ln for ln in lines if 'CIR' not in ln))
        raw = seq.open_seq(path)
        sm0 = raw.seq_model
        assert sm0.do_apertures and sm0.input_ca_list is None
        assert all(ifc.max_aperture == 1.0 for ifc in sm0.ifcs)
        opm = seq.open_seq(path)
        n_set = opm.update_optical_properties(oracle_bundle_fn(opm))
        sm, osp = opm.seq_model, opm.optical_spec
        assert n_set >= sm.get_num_surfaces() - 2
        wvl = sm.central_wavelength()
        for fld in osp.field_of_view.fields:                      # aimed: the chief ray hits the stop centre
            pkg = TR.trace_base(opm, np.array([0., 0.]), fld, wvl, tracer=oracle_tracer)
            assert np.abs(pkg[0][sm.stop_surface][0][:2]).max() < 1e-6      # object at 1e10: start-ray rounding
        heights = np.zeros(sm.get_num_surfaces())
        for fld in osp.field_of_view.fields:                      # every boundary ray passes, some graze
            for pr in osp.pupil.pupil_rays:
                pkg = TR.trace_base(opm, np.array(pr, dtype=float), fld, wvl, tracer=oracle_tracer,
                                    check_apertures=True)
                for i, seg in enumerate(pkg[0]):
                    heights[i] = max(heights[i], np.hypot(seg[0][0], seg[0][1]))
        for i, ifc in enumerate(sm.ifcs[1:-1], start=1):
            if i != sm.stop_surface:
                assert abs(ifc.max_aperture - heights[i]) < 1e-9
        # the same through the reader's do_update switch
        again = seq.open_seq(path, do_update=True, bundle_fn=oracle_bundle_fn(seq.open_seq(path)))
        assert [i.max_aperture for i in again.seq_model.ifcs] == [i.max_aperture for i in sm.ifcs]
    finally:
        os.path.exists(path) and os.remove(path)
    # the sample itself has a CIR record on interface 2: it stays, the others are set
    part = seq.open_seq(part_path)
    assert not part.seq_model.do_apertures and part.seq_model.input_ca_list == [2]
    part.update_optical_properties(oracle_bundle_fn(part))
    assert part.seq_model.ifcs[2].max_aperture == 9.0
    assert all(ifc.max_aperture != 1.0 for ifc in part.seq_model.ifcs[1:-1])
    # a model that stores its apertures (the mirror's own JSON) is left alone
    own = load_model('triplet')
    before = [i.max_aperture for i in own.seq_model.ifcs]
    assert own.update_optical_properties(oracle_bundle_fn(own)) == 0
    assert [i.max_aperture for i in own.seq_model.ifcs] == before
    # Zemax: DIAM kind 0 (automatic semi-diameters) leaves the automatic apertures on
    z = zmx.open_zmx(os.path.join(lens_files(), 'zemax', 'tests', 'US05831776-1.zmx'),
                     glass_map=seq.SubstituteGlasses())
    assert z.seq_model.do_apertures in (True, False) and z.seq_model.ifcs[1].max_aperture != 1.0


def test_set_max_aperture_resizes_clear_apertures_like_the_reference(ref):
    """Surface.set_max_aperture (elem/surface.py:174-179): clear apertures follow, obscurations do not"""
    from rayoptics_b200 import model as M

    def reference_side():
        from oracle import ref_harness as rh
        S = rh.ref().surface
        s = S.Surface()
        s.clear_apertures = [S.Circular(radius=3.0), S.Rectangular(x_half_width=2.0, y_half_width=1.0, x_offset=0.5),
                             S.Circular(radius=0.4, is_obscuration=True)]
        s.set_max_aperture(5.25)
        return (s.max_aperture, (s.clear_apertures[0].radius, s.clear_apertures[2].radius),
                (s.clear_apertures[1].x_half_width, s.clear_apertures[1].y_half_width))
    want_max, want_radii, want_half_widths = ref(reference_side)
    own = M.Surface(clear_apertures=[M.Circular(radius=3.0), M.Rectangular(2.0, 1.0, x_offset=0.5),
                                      M.Circular(radius=0.4, is_obscuration=True)])
    own.set_max_aperture(5.25)
    assert own.max_aperture == want_max == 5.25
    assert (own.clear_apertures[0].radius, own.clear_apertures[2].radius) == want_radii == (5.25, 0.4)
    assert (own.clear_apertures[1].x_half_width, own.clear_apertures[1].y_half_width) == \
           want_half_widths == (5.25, 5.25)


def oracle_tile_fn(opm):
    """tile_fn= seam of vigcalc.set_vig_by_bisection fed by the oracle's grid path"""
    from oracle import rt_oracle
    sm, osp = opm.seq_model, opm.optical_spec
    descs, n_by_wvl, wvls = T.describe_model(sm)

    def fn(fields, wvl, px, py, **opts):
        recs, eprad, z_pupil = osp.grid_fields(fields)
        spec = E.PupilGridSpec(recs, [sm.index_for_wavelength(wvl)], px, py, eprad, z_pupil,
                               apply_vignetting=False, flip_z_dir=sm.z_dir[0], paired=True)
        o = dict(first_surf=1, last_surf=len(descs) - 2)
        o.update(opts)
        return rt_oracle.trace_grid(spec.c_spec(), descs, n_by_wvl, 0, spec.n_rays, _abi.make_opts(**o),
                                    n_threads=4, wvls=wvls)
    return fn


@pytest.mark.parametrize('name', ['dblgauss', 'triplet', 'evenasph', 'rc'])
def test_bisection_vignetting_in_one_launch(name):
    """vigcalc.set_vig_by_bisection (the whole bisection tree of every field and pupil direction
    traced at once) against the sequential calc_vignetted_ray_by_bisection (equal to the
    reference's, test_set_pupil_and_bisection_equal_the_references): same factors, same limiting
    interfaces; the tree holds exactly the positions the search visits."""
    from rayoptics_b200 import vigcalc as V
    a, b = load_model(name), load_model(name)
    for m in (a, b):
        for ifc in m.seq_model.ifcs[1:-1]:
            ifc.set_max_aperture(0.93*ifc.max_aperture)          # so that something limits every direction
        for f in m.optical_spec.field_of_view.fields:
            f.clear_vignetting()
    wvl = a.seq_model.central_wavelength()
    starts = a.optical_spec.pupil.pupil_rays[1:]
    want, want_clip = [], {}
    for fi, fld in enumerate(a.optical_spec.field_of_view.fields):
        row = []
        for di in range(4):
            vig, clip, _ = V.calc_vignetted_ray_by_bisection(a, di//2, np.array(starts[di], dtype=float), fld, wvl,
                                                             tracer=oracle_tracer)
            row.append(vig)
            want_clip[(fi, di)] = clip
        want.append(row)
    clips = V.set_vig_by_bisection(b, oracle_tile_fn(b))
    got = [[f.vux, f.vlx, f.vuy, f.vly] for f in b.optical_spec.field_of_view.fields]
    assert got == want and clips == want_clip
    assert any(v > 0.01 for row in got for v in row)
    tree = V.bisection_tree([0., -1.], 10)
    assert tree.shape == (2047, 2) and tree[0].tolist() == [0., -1.]
    assert tree[1].tolist() == [0., -0.5] and tree[2].tolist() == [0., -1.5]      # blocked / passed
    assert np.all(tree[:, 0] == 0) and len(set(tree[1023:, 1])) == 1024
