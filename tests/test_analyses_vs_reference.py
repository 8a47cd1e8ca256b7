"""RayFan / RayList / RayGrid of rayoptics_b200.analyses against the SAME classes of the
reference (tests/golden/vectors/<model>_analyses.npz: rayoptics.raytr.analyses run unmodified on
a hybrid model with the reference's trace_raw, generator tests/golden/make_golden_analyses.py).

CPU: the classes' host logic (pupil sampling, vignetting, chief ray / reference sphere set-up,
refocus, wave conversion, result shapes) with the tile tracing fed by the oracle through the
`backend=` seam -- bit for bit, OPD included (the oracle keeps libm pow like the reference).
The GPU run of the same comparison is tests/test_zz_gpu_additions.py.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_model
from rayoptics_b200 import _abi, analyses as A, table as T
from refdata import digest, ref  # noqa: F401


class OracleBackend:
    """backend= seam of the analysis classes: chief rays and tiles traced by oracle/rt_oracle.c"""

    def __init__(self, opm):
        from oracle import rt_oracle
        self.o = rt_oracle
        self.descs, self.n_by_wvl, self.wvls = T.describe_model(opm.seq_model)
        self.wide = bool(opm.optical_spec.field_of_view.is_wide_angle)

    def _opts(self, check_apertures):
        # what engine.trace_grid does for RT_PUPIL_WIDE grids (trace_base, trace.py:299-300)
        return _abi.make_opts(first_surf=1, last_surf=len(self.descs) - 2,
                              check_apertures=check_apertures, intersect_obj=not self.wide)

    def chief_rays(self, opt_model, fields, wvls):
        from rayoptics_b200 import engine as E
        osp, sm = opt_model.optical_spec, opt_model.seq_model
        recs, eprad, z_pupil = osp.grid_fields(fields)
        spec = E.PupilGridSpec(recs, [sm.index_for_wavelength(w) for w in wvls], [0.0], [0.0], eprad,
                               z_pupil, apply_vignetting=True, flip_z_dir=sm.z_dir[0])
        p, d, wv, _ = self.o.grid_start_rays(spec.c_spec(), 0, spec.n_rays)
        r = self.o.trace_bundle(self.descs, self.n_by_wvl, p, d, wv, self._opts(False), want_full=True,
                                wvls=self.wvls)
        return r['full'], r['op'], r['status']

    def trace_tile(self, opt_model, spec, want_opd, check_apertures):
        r = self.o.trace_grid(spec.c_spec(), self.descs, self.n_by_wvl, 0, spec.n_rays,
                              self._opts(check_apertures), wvls=self.wvls)
        return {'abr': r['abr'], 'status': r['status'], 'opd': r['opd'] if want_opd else None}


@pytest.mark.parametrize('name', ['dblgauss', 'rc', 'triplet', 'telecentric', 'cellphone', 'fisheye', 'threemir'])
def test_analysis_classes_equal_the_references(name):
    z = np.load(os.path.join(GOLDEN, 'vectors', name + '_analyses.npz'))
    n_fan, n_list, n_grid = (int(x) for x in z['num'])
    opm = load_model(name)
    be = OracleBackend(opm)
    for ci, (f, wl) in enumerate(z['cases']):
        f, wl = int(f), (None if wl < 0 else float(wl))
        for xy in 'xy':
            fan = A.RayFan(opm, f=f, wl=wl, xyfan=xy, num_rays=n_fan, backend=be)
            pup = np.array([p for p, v in fan.fan], dtype=float).reshape(-1, 2)
            val = np.array([v for p, v in fan.fan], dtype=float).reshape(-1, 3)
            assert np.array_equal(pup, z[f'fan{xy}_pupil_{ci}'])
            assert np.array_equal(val, z[f'fan{xy}_vals_{ci}'])
        rl = A.RayList(opm, num_rays=n_list, f=f, wl=wl, backend=be)
        assert np.array_equal(rl.ray_abr, z[f'list_abr_{ci}'])
        rg = A.RayGrid(opm, f=f, wl=wl, num_rays=n_grid, backend=be)
        assert np.array_equal(rg.grid, z[f'grid_{ci}'], equal_nan=True)


def test_functional_forms_equal_the_references(ref):
    """eval_fan / eval_pupil_coords / eval_wavefront / select_plot_data / smooth_plot_data against
    rayoptics.raytr.analyses run on the hybrid model (values stored by tests/refdata.py)"""
    a, b = load_model('dblgauss'), load_model('dblgauss')
    if ref.live:
        from oracle import ref_model
        RT, RA = ref_model.modules()
        H = ref_model.HybridModel(a)
    be = OracleBackend(b)
    fa, fb = a.optical_spec.field_of_view.fields[2], b.optical_spec.field_of_view.fields[2]
    wvl = 656.3

    def keep():
        fa.chief_ray = ((None, None, -1.0), None)        # no re-aiming by the reference
    for xy in (0, 1):
        keep()
        want = ref(lambda: RA.eval_fan(H, fa, wvl, 0.0, xy, num_rays=11))
        got = A.eval_fan(b, fb, wvl, 0.0, xy, num_rays=11, backend=be)
        assert len(want) == len(got)
        for (pw, vw), (pg, vg) in zip(want, got):
            assert tuple(pw) == tuple(pg) and tuple(vw) == tuple(vg)
        for dt in (0, 1, 2):
            xw, yw = ref(lambda: RA.select_plot_data(want, xy, dt))
            xg, yg = A.select_plot_data(got, xy, dt)
            assert np.array_equal(xw, xg) and np.array_equal(yw, yg)
        if xy == 1:
            sw, sg = ref(lambda: RA.smooth_plot_data(xw, yw, 25)), A.smooth_plot_data(xg, yg, 25)
            assert np.array_equal(sw[0], sg[0]) and np.array_equal(sw[1], sg[1])
    keep()
    want = ref(lambda: RA.eval_pupil_coords(H, fa, wvl, 0.0, num_rays=9))
    got = A.eval_pupil_coords(b, fb, wvl, 0.0, num_rays=9, backend=be)
    assert np.array_equal(want, got)
    keep()
    want = ref(lambda: RA.eval_wavefront(H, fa, wvl, 0.0, num_rays=10))
    got = A.eval_wavefront(b, fb, wvl, 0.0, num_rays=10, backend=be)
    assert np.array_equal(want, got, equal_nan=True)
    assert np.array_equal(ref(lambda: fa.ref_sphere[0]), fb.ref_sphere[0])


@pytest.mark.parametrize('name,fi,wvl', [('dblgauss', 2, 656.3), ('telecentric', 1, 587.6),
                                         ('threemir', 1, None), ('cellphone', 4, None), ('fisheye', 3, None),
                                         ('rc', 2, None), ('evenasph', 5, None)])
def test_trace_then_focus_equal_the_references(name, fi, wvl, ref):
    """trace_fan / focus_fan, trace_pupil_coords / focus_pupil_coords, trace_wavefront /
    focus_wavefront (the two-stage forms used for rapid refocus): same traced packages, same
    pre-calculated tuples, same refocused values as rayoptics.raytr.analyses on the hybrid model --
    finite and infinite (telecentric) reference spheres, with defocus and an image shift."""
    from test_trace_drivers import oracle_tracer
    a, b = load_model(name), load_model(name)
    if ref.live:
        from oracle import ref_model
        RT, RA = ref_model.modules()
        H = ref_model.HybridModel(a)
    fa, fb = a.optical_spec.field_of_view.fields[fi], b.optical_spec.field_of_view.fields[fi]
    wvl = a.seq_model.central_wavelength() if wvl is None else wvl
    kw = dict(tracer=oracle_tracer)

    def keep():
        fa.chief_ray = ((None, None, -1.0), None)        # no re-aiming by the reference
    # the traced packages are large: stored as digest() of (pupil, package) rows and of the
    # pre-calculated tuples, which are equal exactly when every number is
    for xy in (0, 1):
        keep()
        if ref.live:
            fw = RA.trace_fan(H, fa, wvl, 0.0, xy, num_rays=9)
        fg = A.trace_fan(b, fb, wvl, 0.0, xy, num_rays=9, **kw)
        assert ref(lambda: len(fw[0])) == len(fg[0]) > 3
        assert ref.digest(lambda: fw[0]) == digest(fg[0])
        assert ref.digest(lambda: fw[1]) == digest(fg[1])
        for foc, delta in ((0.0, None), (0.05, None), (-0.02, np.array([0.001, -0.002]))):
            keep()
            want = ref(lambda: RA.focus_fan(H, fw, fa, wvl, foc, image_delta=delta))
            got = A.focus_fan(b, fg, fb, wvl, foc, image_delta=delta, **kw)
            assert len(want) == len(got)
            for (pw, vw), (pg, vg) in zip(want, got):
                assert tuple(pw) == tuple(pg) and tuple(vw) == tuple(vg)
    # list of pupil coordinates
    pts = [np.array([x, y]) for x in (-0.9, -0.3, 0.0, 0.4, 1.2) for y in (-0.7, 0.0, 0.8)]
    keep()
    if ref.live:
        lw = RA.trace_pupil_coords(H, [p.copy() for p in pts], fa, wvl, 0.0, append_if_none=True)
        ok_w = [r for r in lw if r[2] is not None]
    lg = A.trace_pupil_coords(b, [p.copy() for p in pts], fb, wvl, 0.0, append_if_none=True, **kw)
    assert ref(lambda: len(lw)) == len(lg) == len(pts)
    assert ref(lambda: [r[2] is None for r in lw]) == [r[2] is None for r in lg]
    ok_g = [r for r in lg if r[2] is not None]
    assert ref.digest(lambda: ok_w) == digest(ok_g)
    for foc in (0.0, 0.03):
        keep()
        want = ref(lambda: RA.focus_pupil_coords(H, ok_w, fa, wvl, foc))
        got = A.focus_pupil_coords(b, ok_g, fb, wvl, foc, **kw)
        assert want.shape == got.shape and np.array_equal(want, got)
    # wavefront grid
    keep()
    if ref.live:
        gw = RA.trace_wavefront(H, fa, wvl, 0.0, num_rays=8)
    gg = A.trace_wavefront(b, fb, wvl, 0.0, num_rays=8, **kw)
    assert ref(lambda: [len(row) for row in gw[0]]) == [len(row) for row in gg[0]] == [8]*8
    assert ref(lambda: [[(x, y, p is None) for x, y, p in row] for row in gw[0]]) == \
        [[(x, y, p is None) for x, y, p in row] for row in gg[0]]
    assert ref.digest(lambda: gw[1]) == digest(gg[1])
    for foc, delta in ((0.0, None), (0.04, np.array([0.0005, 0.001]))):
        keep()
        want = ref(lambda: RA.focus_wavefront(H, gw, fa, wvl, foc, image_delta=delta))
        got = A.focus_wavefront(b, gg, fb, wvl, foc, image_delta=delta, **kw)
        assert want.shape == got.shape == (8, 8, 3)
        assert np.array_equal(want, got, equal_nan=True) and np.isfinite(got[:, :, 2]).sum() > 8
    # the one-stage device forms agree with the two-stage host forms to rounding
    be = OracleBackend(b)
    one = A.eval_wavefront(b, fb, wvl, 0.04, image_delta=np.array([0.0005, 0.001]), num_rays=8, backend=be)
    m = np.isfinite(one[:, :, 2])
    assert np.array_equal(m, np.isfinite(got[:, :, 2]))
    assert np.abs(one[:, :, 2][m] - got[:, :, 2][m]).max() < 1e-6
