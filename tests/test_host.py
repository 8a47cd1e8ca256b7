"""CPU: host logic and the C-ABI surface (no compute calls without a GPU)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, MODEL_NAMES, PHASE_MODEL_NAMES, ANGULAR_MODEL_NAMES, load_model
from rayoptics_b200 import _abi, table as T, model as M, engine as E, parallel as P
from refdata import digest, lens_files, ref  # noqa: F401


def test_library_exports_every_declared_symbol():
    """libb200rt.so loads here (no GPU) and exports exactly what include/b200rt.h declares."""
    hdr = open(os.path.join(ROOT, 'include', 'b200rt.h')).read()
    declared = set(re.findall(r'\b(rt_[a-z0-9_]+)\s*\(', hdr))
    assert declared == set(_abi.EXPORTS)
    lib = _abi.load_library()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.rt_abi_version() == _abi.RT_ABI_VERSION
    # a freshly loaded library has counted no launches: asked in a new interpreter, since on a
    # machine with a GPU the tests before this one have launched kernels in this process
    code = 'from rayoptics_b200 import _abi; print(_abi.load_library().rt_launch_count())'
    p = subprocess.run([sys.executable, '-c', code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and p.stdout.strip() == '0', p.stderr[-2000:]


def test_struct_layout_matches_header():
    """ctypes mirrors have the sizes nvcc/gcc give the C structs."""
    from oracle import rt_oracle
    assert rt_oracle.lib().rto_sizeof_surface_desc() == C.sizeof(_abi.rt_surface_desc) == 640
    assert C.sizeof(_abi.rt_opts) == 40
    assert C.sizeof(_abi.rt_out) == 20*8
    assert C.sizeof(_abi.rt_field_desc) == 152


def test_bad_arguments_return_error_codes():
    lib = _abi.load_library()
    handle = C.c_void_p()
    rc = lib.rt_table_create(None, 0, None, 0, 0, C.byref(handle))
    assert rc == -1 and b'rt_table_create' in lib.rt_last_error()
    assert lib.rt_table_destroy(None) == 0
    assert lib.rt_grid_destroy(None) == 0


def test_no_cpu_fallback_when_library_missing(monkeypatch):
    monkeypatch.setattr(_abi, '_lib', None)
    monkeypatch.setattr(_abi, 'LIB_NAME', 'libb200rt_missing.so')
    with pytest.raises(ImportError, match='no CPU fallback'):
        _abi.load_library()


@pytest.mark.parametrize('name', MODEL_NAMES + PHASE_MODEL_NAMES + ANGULAR_MODEL_NAMES + ['telecentric'])
def test_model_roundtrip_and_table(name):
    opm = load_model(name)
    sm = opm.seq_model
    d2 = M.OpticalModel.from_dict(opm.to_dict())
    a, na, _ = T.describe_model(sm)
    b, nb, _ = T.describe_model(d2.seq_model)
    assert bytes(a) == bytes(b) and np.array_equal(na, nb)
    assert len(a) == sm.get_num_surfaces() and na.shape == (len(sm.wvlns), len(a))
    assert a[len(a) - 1].mode == _abi.MODE_IDS['dummy']
    for i, ifc in enumerate(sm.ifcs):
        if type(ifc).__name__ == 'ThinLens':
            assert a[i].profile == _abi.PROFILE_IDS['ThinLens'] and a[i].phase_kind == 1
            assert a[i].phase_obj_pt[2] == ifc.phase_element.obj_pt[2]
            continue
        assert a[i].profile == _abi.PROFILE_IDS[type(ifc.profile).__name__]
        assert a[i].cv == ifc.profile.cv and a[i].max_aperture == ifc.max_aperture


def test_table_accepts_reference_objects(ref):
    """describe_path works on the reference's own Surface/profile objects."""
    opm = load_model('cellphone')
    wvl = opm.seq_model.central_wavelength()
    a, na = T.describe_path(opm.seq_model.path(wvl))

    def on_reference_objects():
        from oracle import ref_harness as rh
        b, nb = T.describe_path(rh.ref_path(opm.seq_model, wvl))
        return bytes(b), nb
    b, nb = ref(on_reference_objects)
    assert bytes(a) == b and na == nb


def test_unsupported_interfaces_are_rejected():
    class ThinLens:           # reference: oprops/thinlens.py (no profile, phase element)
        interact_mode = 'transmit'
        phase_element = object()
    with pytest.raises(T.UnsupportedInterfaceError):
        T.describe_path([(ThinLens(), None, None, 1.0, 1)])


def test_accumulated_steps_is_the_reference_loop():
    """start += step repeated, NOT linspace (raytr/trace.py:567-604)."""
    xs = E.accumulated_steps(-1.0, 1.0, 512)
    start = np.array([-1.0, -1.0])
    step = np.array((np.array([1.0, 1.0]) - start)/(512 - 1))
    ref = []
    for _ in range(512):
        ref.append(start[0])
        start[0] += step[0]
    assert np.array_equal(xs, np.array(ref))
    assert not np.array_equal(xs, np.linspace(-1, 1, 512))


@pytest.mark.parametrize('name', ['dblgauss', 'rc', 'cellphone', 'singlet'])
def test_start_rays_numpy_vs_oracle(oracle, name):
    """ray_start_from_osp evaluated by numpy (the reference's expressions) and
    the C restatement used by the oracle / mirrored by the grid kernel agree
    bit for bit, including vignetting and the accumulated pupil steps."""
    opm = load_model(name)
    osp, sm = opm.optical_spec, opm.seq_model
    num = 9
    spec = E.grid_spec_for_model(opm, num)
    p, d, wv, pup = oracle.grid_start_rays(spec.c_spec(), 0, spec.n_rays)
    xs = E.accumulated_steps(-1.0, 1.0, num)
    k = 0
    for fld in osp.fov.fields:
        for wi in range(len(sm.wvlns)):
            for i in range(num):
                for j in range(num):
                    pupil = fld.apply_vignetting(np.array([xs[i], xs[j]]))
                    pt0, dir0 = osp.ray_start_from_osp(pupil, fld, 'rel pupil')
                    if dir0[2]*sm.z_dir[0] < 0:
                        dir0 = -dir0
                    assert np.array_equal(pup[:, k], pupil)
                    assert np.array_equal(p[:, k], pt0) and np.array_equal(d[:, k], dir0)
                    assert wv[k] == wi
                    k += 1
    assert k == spec.n_rays


def test_grid_geometry():
    opm = load_model('dblgauss')
    spec = E.grid_spec_for_model(opm, 100)
    assert spec.n_rays == 9*100*100 and spec.chunks_per_tile == 40 and spec.n_chunks == 360
    assert spec.first_ray_of_chunk(0) == 0 and spec.first_ray_of_chunk(40) == 10000
    assert spec.first_ray_of_chunk(39) == 39*256 and spec.rays_in_chunks(39, 41) == 10000 - 39*256 + 256
    assert spec.rays_in_chunks(0, spec.n_chunks) == spec.n_rays


def test_shard_chunks_partitions_exactly():
    for n in (0, 1, 7, 360, 9216, 1000003):
        for world in (1, 2, 3, 4, 8):
            edges = [P.shard_chunks(n, r, world) for r in range(world)]
            assert edges[0][0] == 0 and edges[-1][1] == n
            for (a, b), (c, d) in zip(edges[:-1], edges[1:]):
                assert b == c and a <= b
            sizes = [b - a for a, b in edges]
            assert max(sizes) - min(sizes) <= 1


def test_first_order_against_stored_reference_values():
    """Chief-ray aim points stored by the reference in its .roa files pin
    first-order data + aiming (SURVEY.md 8(c)): Sasian triplet 20 deg field."""
    opm = load_model('triplet')
    aim = opm.optical_spec.fov.fields[1].aim_info
    assert aim[1] == pytest.approx(-0.3143052528206426, abs=1e-12)
    fod = opm.optical_spec.fod
    assert fod.efl == pytest.approx(50.0, rel=2e-4)
    assert load_model('dblgauss').optical_spec.fod.efl == pytest.approx(100.0, rel=2e-4)


def _same_prescription(a, b, skip_modes=()):
    """two SequentialModel mirrors describe the same path (all wavelengths)"""
    assert a.wvlns == pytest.approx(b.wvlns, rel=1e-15) and a.get_num_surfaces() == b.get_num_surfaces()
    for wa, wb in zip(a.wvlns, b.wvlns):
        da, na = T.describe_path(a.path(wa))
        db, nb = T.describe_path(b.path(wb))
        assert na == nb
        for i, (x, y) in enumerate(zip(da, db)):
            assert (x.profile, x.cv, x.cc, list(x.coefs), list(x.t), x.z_dir) == \
                   (y.profile, y.cv, y.cc, list(y.coefs), list(y.t), y.z_dir)
            assert x.mode == y.mode or i in skip_modes


def test_seq_reader():
    """CODE V .seq reader (codev/cmdproc.py:56-449): own sample, and the reference's double Gauss
    (same table as the numeric fixture)."""
    from rayoptics_b200 import seq
    m = seq.open_seq(os.path.join(ROOT, 'tests', 'golden', 'samples', 'triplet_fict.seq'))
    sm, osp = m.seq_model, m.optical_spec
    assert m.name == 'fictitious triplet' and sm.get_num_surfaces() == 9 and sm.stop_surface == 4
    assert sm.ifcs[1].profile.cv == 1/21.25 and sm.gaps[1].thi == 5.0          # radius mode
    assert type(sm.ifcs[3].profile).__name__ == 'EvenPolynomial' and sm.ifcs[3].profile.cc == -0.25
    assert sm.ifcs[3].profile.coefs[:3] == [0.0, 1.5e-6, -2.0e-9]              # A -> r**4
    assert sm.gaps[1].medium.rindex(587.5618) == pytest.approx(1.620, abs=1e-9)   # 620.603
    assert sm.ifcs[2].max_aperture == 9.0 and sm.wvlns == [656.3, 587.6, 486.1] and sm.ref_wvl == 1
    assert osp.pupil.key == ('image', 'f/#') and osp.fod.fno == pytest.approx(4.5, rel=1e-12)
    assert [(f.y, f.vuy, f.vly) for f in osp.field_of_view.fields] == \
        [(0.0, 0.0, 0.0), (7.0, 0.05, 0.05), (10.0, 0.1, 0.15)]
    assert osp.defocus.focus_shift == -0.05
    T.describe_model(sm)                                   # compiles into a surface table
    with pytest.raises(KeyError):
        seq._medium('NLASF99_SCHOTT', {})            # not among the built-in 17
    fx = load_model('dblgauss').seq_model
    gm = {'NSSK2_SCHOTT': fx.gaps[1].medium, 'NSK2_SCHOTT': fx.gaps[3].medium,
          'F5_SCHOTT': fx.gaps[4].medium, 'NSK16_SCHOTT': fx.gaps[8].medium}
    o = seq.open_seq(os.path.join(lens_files(), 'codev', 'tests', 'ag_dblgauss.seq'), glass_map=gm)
    o.seq_model.gaps[-1].thi += o.optical_spec.defocus.focus_shift   # the fixture lumps the defocus
    o.update_model()
    _same_prescription(o.seq_model, fx, skip_modes=(0, 6))
    assert o.optical_spec.fod.efl == pytest.approx(100.0038, abs=1e-4)      # .lis: EFL 100.0038


def test_zmx_reader():
    """Zemax .zmx reader (zemax/zmxread.py:93-388) on the file the `evenasph` fixture was
    transcribed from."""
    import glob
    from rayoptics_b200 import zmx
    hits = [f for f in glob.glob(os.path.join(lens_files(), 'zemax', 'tests', '*')) if 'US08427765-1' in f]
    assert hits
    glass = {'J-LAK14': (1.6968, 55.5), 'L-TIM28': (1.68893, 31.1), 'SF11': (1.78472, 25.7),
             'TAF3': (1.8042, 46.5), 'TAFD30': (1.883, 40.8)}
    m = zmx.open_zmx(hits[0], glass_map=glass)
    fx = load_model('evenasph')
    _same_prescription(m.seq_model, fx.seq_model, skip_modes=(5,))
    assert m.seq_model.stop_surface == 5 and m.optical_spec.pupil.key == ('image', 'f/#')
    assert [f.y for f in m.optical_spec.field_of_view.fields] == [0.0, 8.0, 13.6]
    with pytest.raises(KeyError):
        zmx.open_zmx(hits[0], glass_map={})


def test_small_raytrace_helpers_match_reference(ref):
    """bend / reflect / calc_optical_path of rayoptics_b200.raytrace against the reference's"""
    from oracle import ref_harness as rh
    from rayoptics_b200 import raytrace as RT
    if ref.live:
        R = rh.ref().raytrace

    def ref_bend(d, n, n_in, n_out):            # None: the reference raised TraceTIRError
        try:
            return R.bend(d, n, n_in, n_out)
        except rh.ref().traceerror.TraceTIRError:
            return None
    rng = np.random.default_rng(2)
    for _ in range(200):
        d = rng.standard_normal(3); d /= np.linalg.norm(d)
        n = rng.standard_normal(3); n /= np.linalg.norm(n)
        assert np.array_equal(RT.reflect(d, n), ref(lambda: R.reflect(d, n)))
        n_in, n_out = rng.uniform(1, 2, 2)
        want = ref(lambda: ref_bend(d, n, n_in, n_out))
        if want is None:
            with pytest.raises(RT.TraceTIRError):
                RT.bend(d, n, n_in, n_out)
        else:
            assert np.array_equal(RT.bend(d, n, n_in, n_out), want)
    opm = load_model('triplet')
    sm = opm.seq_model
    wvl = sm.central_wavelength()
    r = ref(lambda: rh.ref_trace(rh.ref_path(sm, wvl), [0., 1., 0.], [0., 0., 1.], wvl, first_surf=1,
                                 last_surf=sm.get_num_surfaces() - 2))
    ray = [[s[0:3], s[3:6], s[6], s[7:10]] for s in r['ray']]
    path = list(sm.path(wvl))
    assert RT.calc_optical_path(ray, path) == ref(lambda: R.calc_optical_path(ray, iter(rh.ref_path(sm, wvl))))


def test_samplers_match_reference(ref):
    """rayoptics_b200/sampler.py against rayoptics.raytr.sampler (importable)"""
    import importlib
    from rayoptics_b200 import sampler as S
    if ref.live:
        from oracle import ref_harness as rh
        rh.ref()
        RS = importlib.import_module('rayoptics.raytr.sampler')

    def rng():
        return [np.array([-1., -0.5]), np.array([1., 0.75]), 11]
    # the sample sequences are compared as digest(): equal exactly when every sample is
    for name in ('grid_ray_generator', 'csd_grid_ray_generator', 'polar_grid_ray_generator'):
        b = list(getattr(S, name)(rng()))
        assert len(b) == 121 and digest(b) == ref.digest(lambda: list(getattr(RS, name)(rng())))
    b = [z.copy() for z in S.R_2_quasi_random_generator(50)]
    assert digest(b) == ref.digest(lambda: [z.copy() for z in RS.R_2_quasi_random_generator(50)])
    assert S.phi(2) == ref(lambda: RS.phi(2))
    b = list(S.create_generator(S.R_2_quasi_random_generator, 20, mapper=S.concentric_sample_disk))
    assert digest(b) == ref.digest(
        lambda: list(RS.create_generator(RS.R_2_quasi_random_generator, 20, mapper=RS.concentric_sample_disk)))
    # whole-array producers == the reference's per-sample generators, bit for bit
    for num in (2, 21, 64):
        g = lambda: [np.array([-1., -1.]), np.array([1., 1.]), num]      # noqa: E731
        sq, dk = S.square_grid_points(g()), S.disk_grid_points(g())
        assert sq.shape == dk.shape == (num*num, 2)
        assert digest(sq) == ref.digest(lambda: np.array(list(RS.grid_ray_generator(g()))))
        assert digest(dk) == ref.digest(lambda: np.array(list(RS.csd_grid_ray_generator(g()))))
        xs, ys = S.square_grid_axes(g())
        assert np.array_equal(S.square_grid_points(g()).reshape(num, num, 2)[:, 0, 0], xs)
    u = np.array([[0., 0.], [0.5, 0.5], [1., 0.], [0., 1.], [0.25, 0.75], [0.75, 0.25], [0.3, 0.3],
                  [0.5, 0.1], [0.1, 0.5]])
    for off in (True, False):
        want = ref(lambda: np.array([RS.concentric_sample_disk(x, offset=off) for x in u], dtype=float))
        assert np.array_equal(S.concentric_disk(u, offset=off), want)
    r2 = S.r2_sequence(500)
    assert r2.shape == (500, 2)
    assert digest(r2) == ref.digest(lambda: np.array([z.copy() for z in RS.R_2_quasi_random_generator(500)]))


def test_psf_helpers_match_reference(ref):
    """psf_sampling / calc_psf_scaling against rayoptics.raytr.analyses (importable)"""
    from rayoptics_b200 import analyses as A
    if ref.live:
        from oracle import ref_model
        RT, RA = ref_model.modules()
    for args in ((None, 32, 8), (128, None, 8), (128, 32, None)):
        assert A.psf_sampling(*args) == ref(lambda: RA.psf_sampling(*args))
    opm = load_model('dblgauss')
    fld = opm.optical_spec.field_of_view.fields[1]
    fld.ref_sphere = (np.zeros(3), np.array([0., 0., 1.]), 123.456, None)
    assert A.calc_psf_scaling(opm, fld, 587.6, 32, 128) == ref(lambda: RA.calc_psf_scaling(opm, fld, 587.6, 32, 128))


def test_table_cache_key_sees_in_place_edits():
    """The drop-in's table cache (raytrace._table_for_path, analyses._table_for) is keyed on
    the compiled descriptor records: editing a clear aperture, a conic constant or a
    polynomial coefficient in place -- without update_model(), whose cache clearing
    (seq/sequential.py:666-668) is the reference's own invalidation point -- gives a new key."""
    from rayoptics_b200 import raytrace as RT
    opm = load_model('exotic')
    sm = opm.seq_model
    segs = lambda: list(sm.path(sm.central_wavelength()))       # noqa: E731
    k0 = RT._fingerprint(segs())
    assert RT._fingerprint(segs()) == k0
    seen = {k0}

    def changed():
        k = RT._fingerprint(segs())
        assert k not in seen
        seen.add(k)

    ifc_ca = next(i for i in sm.ifcs if getattr(i, 'clear_apertures', None))
    ca = ifc_ca.clear_apertures[0]
    for attr in ('radius', 'x_half_width', 'y_half_width'):
        if hasattr(ca, attr):
            setattr(ca, attr, getattr(ca, attr)*1.25)
            changed()
    ca.x_offset += 0.125
    changed()
    ca.y_offset -= 0.25
    changed()
    ca.is_obscuration = not getattr(ca, 'is_obscuration', False)
    changed()
    ifc_poly = next(i for i in sm.ifcs if len(getattr(i.profile, 'coefs', [])) > 0)
    ifc_poly.profile.coefs[0] += 1e-9
    changed()
    ifc_cc = next(i for i in sm.ifcs if hasattr(i.profile, 'cc'))
    ifc_cc.profile.cc = ifc_cc.profile.cc - 0.5
    if hasattr(ifc_cc.profile, 'update'):
        ifc_cc.profile.update()
    changed()
    sm.ifcs[1].max_aperture *= 2.0
    changed()
    sm.ifcs[1].interact_mode = 'reflect'
    changed()
    sm.ifcs[2].profile.cv += 1e-6
    changed()
    rt, t = sm.lcl_tfrms[2]
    sm.lcl_tfrms[2] = (rt, t + np.array([0., 1e-3, 0.]))
    changed()
    sm.lcl_tfrms[3] = (np.ascontiguousarray(sm.lcl_tfrms[3][0].T).T.copy(order='F')
                       if sm.lcl_tfrms[3][0].flags['C_CONTIGUOUS'] else np.ascontiguousarray(sm.lcl_tfrms[3][0]),
                       sm.lcl_tfrms[3][1])
    if not np.array_equal(sm.lcl_tfrms[3][0], np.identity(3)):
        changed()                          # same numbers, other memory order: other dgemv rounding
    # and the key is complete with respect to what the table is compiled from: equal keys <=> equal
    # descriptor bytes over all fixture models
    seen_keys = {}
    for name in MODEL_NAMES + PHASE_MODEL_NAMES + ANGULAR_MODEL_NAMES:
        m = load_model(name).seq_model
        for w in m.wvlns:
            p = list(m.path(w))
            descs, ns = T.describe_path(p)
            assert seen_keys.setdefault(RT._fingerprint(p), (bytes(descs), tuple(ns))) == (bytes(descs), tuple(ns))


def test_nan_status_decoding():
    """engine.decode_nan_status: the payload convention of RT_OUT_ABR_NAN_STATUS (include/b200rt.h)."""
    base = _abi.RT_NAN_PAYLOAD_BASE
    bits = np.array([[0, base | 3, base | 1, base | 5], [0, base | 12, base | 0, base | 7]], dtype=np.uint64)
    abr = bits.view(np.float64).copy()
    abr[:, 0] = [0.25, -0.5]
    st, fs = E.decode_nan_status(abr)
    assert st.tolist() == [0, 3, 1, 5] and fs.tolist() == [-1, 12, 0, 7]
    assert np.isnan(abr[:, 1:]).all()


def test_tilts_and_decenters_against_the_codev_listing(oracle):
    """Decenter / tilt convention pinned by an external known answer: the reference ships CODE V's
    ray listing (codev/tests/threemrc.lis) of its three-mirror test lens, whose every surface is
    decentered and tilted ('dec and return').  Rays of the fixture model (read from the same .seq by
    rayoptics_b200/seq.py: DecenterData, Euler rotation, forward transforms) land on the listed
    coordinates to the listing's 6 decimals."""
    import json
    kat = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'kat.json')))['threemir_lis']
    opm = load_model('threemir')
    sm = opm.seq_model
    assert sum(1 for ifc in sm.ifcs if ifc.decenter is not None) == 5
    descs, n_by_wvl, wvls = T.describe_model(sm)
    opts = _abi.make_opts(first_surf=1, last_surf=len(descs) - 2)
    for ray in kat['rays']:
        p0 = np.array([[0.], [ray['y0']], [0.]])
        d0 = np.array([[0.], [0.], [1.]])
        r = oracle.trace_bundle(descs, n_by_wvl, p0, d0, np.zeros(1, np.int32), opts, want_full=True)
        assert r['status'][0] == 0
        got = r['full'][1:6, 0:3, 0]
        assert np.abs(got - np.array(ray['xyz'])).max() < kat['abs_tol']
        d = r['full'][1:6, 3:6, 0]
        assert np.abs(d[:, 1]/d[:, 2] - np.array(ray['tan_y'])).max() < kat['abs_tol']


def test_seq_reader_tilt_commands():
    """XDE YDE ZDE ADE BDE CDE DAR BEN REV (codev/cmdproc.py:544-576) on the reference's own tilt test
    files: fold mirrors ('bend') keep the axial ray on every vertex, and the decenter / reverse pairs
    bring it back onto the axis -- what those files were written to show."""
    from rayoptics_b200 import seq
    from oracle import rt_oracle
    base = os.path.join(lens_files(), 'codev', 'tests')
    for name, on_vertex, on_axis in (('dec_tilt_test.seq', True, True), ('tilt_test.seq', False, False),
                                     ('dec_test.seq', False, True), ('dec_rev_tilt_test.seq', False, True),
                                     ('dar_test.seq', False, True)):
        opm = seq.open_seq(os.path.join(base, name))
        descs, n_by_wvl, wvls = T.describe_model(opm.seq_model)
        r = rt_oracle.trace_bundle(descs, n_by_wvl, np.zeros((3, 1)), np.array([[0.], [0.], [1.]]),
                                   np.zeros(1, np.int32),
                                   _abi.make_opts(first_surf=1, last_surf=len(descs) - 2), want_full=True)
        assert r['status'][0] == 0
        pts, dirs = r['full'][:, 0:3, 0], r['full'][:, 3:6, 0]
        assert abs(abs(dirs[-1, 2]) - 1.0) < 1e-12
        if on_axis:
            assert np.abs(pts[-1, 0:2]).max() < 1e-9
        else:                                   # tilt_test.seq: 100 mm along a 45 degree leg
            assert abs(pts[-1, 1] + 100.0*np.sin(np.pi/4)) < 1e-9
        if on_vertex:
            assert np.abs(pts).max() < 1e-9
    d = opm.seq_model.ifcs[2].decenter                      # dar_test.seq: YDE 1; ADE 45; DAR
    assert d.dtype == 'dec and return' and d.dec[1] == 1.0 and d.euler[0] == 45.0
    m2 = M.OpticalModel.from_dict(opm.to_dict())            # decenters survive the JSON round trip
    for (ra, ta), (rb, tb) in zip(opm.seq_model.lcl_tfrms, m2.seq_model.lcl_tfrms):
        assert np.array_equal(ra, rb) and np.array_equal(ta, tb)
        assert ra.flags['C_CONTIGUOUS'] == rb.flags['C_CONTIGUOUS']


def test_zmx_reader_coordinate_breaks():
    """COORDBRK surfaces (zemax/zmxread.py:314-316,341-355) of the reference's own Zemax test files:
    phantom interfaces with DecenterData; the folded system of HoO-V2C18Ex66 (9 coordinate breaks)
    brings the axial ray back onto the axis, direction (0, 0, 1)."""
    from rayoptics_b200 import zmx
    from oracle import rt_oracle
    base = os.path.join(lens_files(), 'zemax', 'tests')
    opm = zmx.open_zmx(os.path.join(base, 'HoO-V2C18Ex66.zmx'),
                       glass_map={'BK7': (1.5168, 64.17), 'SF2': (1.64769, 33.85), 'F2': (1.62004, 36.37),
                                  'SK16': (1.62041, 60.32), 'N-BK7': (1.5168, 64.17), 'SILICA': (1.4585, 67.8),
                                  'SF5': (1.6727, 32.2), 'BAK4': (1.5688, 56.1), 'SF1': (1.71736, 29.5),
                                  'K5': (1.52249, 59.5), 'SK2': (1.60738, 56.65), 'LAK9': (1.691, 54.7)})
    sm = opm.seq_model
    cb = [i for i in sm.ifcs if i.decenter is not None]
    assert len(cb) == 9 and all(i.interact_mode == 'phantom' for i in cb)
    assert any(i.decenter.dtype == 'reverse' for i in cb) or all(i.decenter.dtype == 'decenter' for i in cb)
    descs, n_by_wvl, _ = T.describe_model(sm)
    r = rt_oracle.trace_bundle(descs, n_by_wvl, np.zeros((3, 1)), np.array([[0.], [0.], [1.]]),
                               np.zeros(1, np.int32), _abi.make_opts(first_surf=1, last_surf=len(descs) - 2))
    assert r['status'][0] == 0
    assert np.abs(r['last'][0:2, 0]).max() < 1e-9 and abs(r['last'][5, 0] - 1.0) < 1e-12


def test_weighted_sharding():
    """parallel.shard_chunks_weighted: ranges tile the chunk space, equal weights reproduce the
    plain split to within a chunk, and unequal weights equalise the work."""
    cpt, n_tiles = 64, 9
    w = np.ones(n_tiles)
    cuts = [P.shard_chunks_weighted(cpt, w, r, 4) for r in range(4)]
    assert cuts[0][0] == 0 and cuts[-1][1] == cpt*n_tiles
    assert all(a[1] == b[0] for a, b in zip(cuts[:-1], cuts[1:]))
    assert all(abs((e - b) - cpt*n_tiles/4) <= 1 for b, e in cuts)
    w = np.array([1.0, 1.0, 1.0, 0.5, 0.5, 0.5, 0.25, 0.25, 0.25])
    cuts = [P.shard_chunks_weighted(cpt, w, r, 3) for r in range(3)]
    work = [np.repeat(w, cpt)[b:e].sum() for b, e in cuts]
    assert max(work)/min(work) < 1.02 and cuts[0][1] - cuts[0][0] < cuts[2][1] - cuts[2][0]
    summ = np.zeros((2, 16)); summ[0, 0] = 100; summ[1, 0] = 50; summ[1, 3] = 50
    assert P.weights_from_summary(summ).tolist() == [100.0, 65.0]


def test_local_transforms_equal_the_references(ref):
    """model.DecenterData / forward_transform / compute_local_transforms against the reference's own
    elem/surface.py:274-337 + elem/transform.py:79-166 on random decenter sets (all four dtypes):
    same rotation matrices, translations AND numpy memory layouts (which decide the dgemv rounding of
    the trace, table.py has_tfrm).  transforms3d is not installed: the reference's euler2rot3d gets
    this package's restatement of `euler2mat(..., 'rxyz')` through the ref_harness stand-in module,
    so what is compared is everything around it; the rotation itself is pinned by the CODE V listing."""
    import importlib
    import sys
    import types
    if ref.live:
        from oracle import ref_harness as rh
        R = rh.ref()
        t3 = sys.modules['transforms3d']
        t3.euler.euler2mat = lambda ai, aj, ak, axes='rxyz': M.euler2mat_rxyz(ai, aj, ak)
        RT = importlib.import_module('rayoptics.elem.transform')
        S = R.surface

    def with_layout(tfrms):                         # the memory layouts are part of what is compared
        return [(r, t, r.flags['C_CONTIGUOUS'], r.flags['F_CONTIGUOUS']) for r, t in tfrms]
    rng = np.random.default_rng(5)
    dtypes = ['decenter', 'reverse', 'dec and return', 'bend']
    for trial in range(40):
        n = int(rng.integers(3, 9))
        own, their_ifcs, thi = [], [], rng.uniform(-30, 60, n - 1)
        decs = []
        for i in range(n):
            so = M.Surface()
            decs.append(None)
            if rng.random() < 0.6:
                dt = dtypes[int(rng.integers(4))]
                vals = [float(v) if rng.random() < 0.7 else 0.0 for v in rng.uniform(-20, 20, 5)]
                so.decenter = M.DecenterData(dt, *vals)
                decs[-1] = (dt, vals)
            own.append(so)
        if ref.live:
            for dec in decs:
                sr = S.Surface()
                if dec is not None:
                    sr.decenter = S.DecenterData(dec[0], *dec[1])
                    sr.decenter.update()
                their_ifcs.append(sr)
        gaps = [M.Gap(float(t)) for t in thi]
        # (rotation, translation, C / F layout) of every interface, compared as digest()
        mine = M.compute_local_transforms(own, gaps)
        seq = types.SimpleNamespace(ifcs=their_ifcs, gaps=gaps, get_num_surfaces=lambda: n)
        assert len(mine) == n
        assert digest(with_layout(mine)) == ref.digest(lambda: with_layout(RT.compute_local_transforms(seq, None, 1)))
        back = M.compute_local_transforms(own, gaps, step=-1)          # image -> object paths
        assert len(back) == n
        assert digest(with_layout(back)) == ref.digest(lambda: with_layout(RT.compute_local_transforms(seq, None, -1)))
        # global coordinates w.r.t. a random interface, with and without an origin transform
        seq.z_dir = [1]*(n - 1)
        glo = int(rng.integers(0, n - 1))
        origin = None if trial % 2 else (M.euler2mat_rxyz(0.1, -0.2, 0.05), np.array([1., -2., 3.]))
        mine = M.compute_global_coords(own, gaps, glo, origin)
        assert len(mine) == n and digest(mine) == ref.digest(lambda: RT.compute_global_coords(seq, glo, origin))


def test_builtin_glass_table():
    """glass names resolve without a glass_map for the catalog glasses the reference's lens files
    carry; N-BK7 gives the datasheet n_d; unknown names still raise."""
    from rayoptics_b200 import seq
    assert abs(seq._medium('N-BK7', None).rindex(587.5618) - 1.5168) < 2e-6
    assert abs(seq._medium('n-lak9_schott', {}).rindex(587.5618) - 1.6910) < 2e-5
    assert seq._medium('N-BK7', {'N-BK7': 1.5}).rindex(500.0) == 1.5          # the caller's map wins
    with pytest.raises(KeyError, match='glass_table'):
        seq._medium('NOT-A-GLASS', None)


def test_seq_reader_private_catalog_and_doe():
    """CODV_65988.seq (the reference's hybrid-asphere import test): '&' continuation lines, a private
    catalog glass (PRV / PWL / END -> tabulated index), and a diffractive surface (DIF DOE, HOR, HWL,
    HCT R, HCO C1; codev/cmdproc.py:579-618) compiled into the table as a radial DOE."""
    from rayoptics_b200 import seq
    path = os.path.join(lens_files(), 'codev', 'tests', 'CODV_65988.seq')
    opm = seq.open_seq(path)
    sm = opm.seq_model
    assert sm.get_num_surfaces() == 4 and sm.wvlns == [656.2725, 587.5618, 486.1327]
    med = sm.gaps[1].medium
    assert type(med).__name__ == 'TableIndex' and med.rindex(587.6) == 1.53116 and med.rindex(486.1) == 1.5378
    assert 1.527 < med.rindex(656.2725) < 1.5286                  # between the 700 and 650 nm entries
    pe = sm.ifcs[1].phase_element
    assert (type(pe).__name__, pe.coefficients, pe.ref_wl, pe.order) == \
        ('DiffractiveElement', [-0.001807322521767816], 587.5618, 1.0)
    prf = sm.ifcs[1].profile
    assert type(prf).__name__ == 'EvenPolynomial' and prf.cc == -0.71
    assert prf.coefs[1:4] == [-0.1581980090969e-4, -0.2770951746068999e-6, -0.1216086045095e-8]
    descs, n_by_wvl, _ = T.describe_model(sm)
    assert descs[1].phase_kind == _abi.PHASE_IDS['DiffractiveElement'] and descs[1].n_phase_coefs == 1


def test_zmx_reader_paraxial_and_grating(tmp_path):
    """PARAXIAL -> ThinLens(power = 1/PARM1), DGRATING -> DiffractionGrating(PARM1 lines/um, PARM2 order)
    (zemax/zmxread.py:317-324,356-366); both compile into the table."""
    from rayoptics_b200 import zmx
    text = '\n'.join([
        'UNIT MM X W X CM MR CPMM', 'ENPD 10', 'WAVM 1 0.55 1', 'FTYP 0 0 1 1 0 0 0', 'XFLN 0', 'YFLN 0',
        'SURF 0', ' TYPE STANDARD', ' CURV 0', ' DISZ INFINITY',
        'SURF 1', ' STOP', ' TYPE PARAXIAL', ' CURV 0', ' DISZ 5', ' PARM 1 100', ' DIAM 5',
        'SURF 2', ' TYPE DGRATING', ' CURV 0', ' DISZ 95', ' PARM 1 0.3', ' PARM 2 1', ' DIAM 5',
        'SURF 3', ' TYPE STANDARD', ' CURV 0', ' DISZ 0'])
    f = tmp_path / 'thin.zmx'
    f.write_text(text)
    opm = zmx.open_zmx(str(f))
    sm = opm.seq_model
    assert type(sm.ifcs[1]).__name__ == 'ThinLens' and sm.ifcs[1].optical_power == 0.01
    g = sm.ifcs[2].phase_element
    assert type(g).__name__ == 'DiffractionGrating' and g.order == 1 and g.grating_lpmm == 0.3*1000
    descs, _, _ = T.describe_model(sm)
    assert descs[1].profile == _abi.PROFILE_IDS['ThinLens'] and descs[2].phase_kind == _abi.PHASE_IDS['DiffractionGrating']


def test_seq_tokenizer_known_answers():
    """The reference's own tokenizer tests (codev/tests/test_reader.py:6-45: continuation lines,
    ';' commands, '!' comments, blanks as delimiters, quoted strings) applied to seq._commands."""
    from rayoptics_b200 import seq

    def toks(lines):
        return [[t.strip('\'"') for t in cmd] for cmd in seq._commands('\n'.join(lines))]
    assert toks(['ab&', 'cd&', 'ef', 'gh']) == [['abcdef'], ['gh']]
    assert toks(['ab; cd!ef; gh']) == [['ab'], ['cd']]
    assert toks(['ab; cd; ef', 'gh;ij& ', 'kl; mn']) == [['ab'], ['cd'], ['ef'], ['gh'], ['ijkl'], ['mn']]
    assert toks(['s &', '.07 10 ', 's & ', ' 0 .001']) == [['s', '.07', '10'], ['s', '0', '.001']]
    assert toks(['tit "this is a title"', ' ! this is a comment line', 'dim m', 'so 0 1e11 ! infinite object']) == \
        [['tit', 'this is a title'], ['dim', 'm'], ['so', '0', '1e11']]
    assert toks([]) == [] and toks(['', '! this comment will be stripped out', '', '    ! so will this one']) == []


def test_seq_reader_units_and_laurent_glass(tmp_path):
    """DIM I / C (codev/cmdproc.py:281-289, SystemSpec.nm_to_sys_units incl. its pass-through for the
    importer's 'inches'), a private-catalog glass given by Laurent coefficients, and CODE V's hyphen-less
    catalog names (NBK7_SCHOTT) resolved through the built-in table."""
    from rayoptics_b200 import seq
    f = tmp_path / 'u.seq'
    f.write_text('\n'.join([
        'RDM', 'DIM I', 'EPD 1', 'WL 587.6', 'PRV', ' PWL 550.0',
        " 'NOA61' LAU 2.36390625 0.0 0.025493134 -0.000580235 -0.349933e-5 0.445404e-7", 'END',
        'SO 0 1e11', "S 10 0.2 'NOA61'", ' STO', 'S -10 0.1 NBK7_SCHOTT', 'S 0 9', 'SI 0 0']))
    opm = seq.open_seq(str(f))
    assert opm.dimensions == 'inches' and opm.nm_to_sys_units(500.0) == 500.0
    n = opm.seq_model.gaps[1].medium.rindex(587.5618)
    assert abs(n - 1.5597) < 2e-4                                  # NOA61: n_d = 1.56
    assert abs(opm.seq_model.gaps[2].medium.rindex(587.5618) - 1.5168) < 2e-6
    assert M.OpticalModel.from_dict(opm.to_dict()).dimensions == 'inches'
    opm.dimensions = 'cm'
    assert opm.nm_to_sys_units(500.0) == 1e-7*500.0


@pytest.mark.parametrize('name', MODEL_NAMES + PHASE_MODEL_NAMES + ANGULAR_MODEL_NAMES + ['telecentric'])
def test_table_validation_accepts_every_fixture_without_a_gpu(name):
    """rt_table_create validates the descriptors BEFORE its first CUDA call, so the validation
    is testable here: every fixture model (gratings, radial DOEs, holograms, toroids ...) must get past
    it -- on a machine without a GPU that means the call then fails with RT_ERR_CUDA (-2), never with
    RT_ERR_UNSUPPORTED (-3) / RT_ERR_INVALID (-1) -- and broken descriptors must be refused by it.
    (Round 1 shipped a validation that rejected the grating / DOE kinds; only the GPU run showed it.)"""
    import torch
    if torch.cuda.is_available():
        pytest.skip('needs a machine WITHOUT a CUDA device (the call would succeed)')
    lib = _abi.load_library()
    descs, n_by_wvl, _ = T.describe_model(load_model(name).seq_model)
    n_by_wvl = np.ascontiguousarray(n_by_wvl)
    h = C.c_void_p()

    def create(d):
        return lib.rt_table_create(d, len(d), n_by_wvl.ctypes.data_as(_abi.c_double_p),
                                   n_by_wvl.shape[0], 0, C.byref(h))
    assert create(descs) == -2, lib.rt_last_error()
    for field, bad, want in (('phase_kind', 9, -3), ('profile', 11, -3), ('mode', 7, -3),
                             ('n_coefs', _abi.RT_MAX_COEFS + 1, -1), ('n_apertures', 9, -1),
                             ('n_phase_coefs', _abi.RT_MAX_PHASE_COEFS + 1, -1)):
        broken = (type(descs[0])*len(descs))(*descs)
        setattr(broken[1], field, bad)
        assert create(broken) == want, (field, lib.rt_last_error())


@pytest.mark.parametrize('name', ['dblgauss', 'relay_na', 'relay_fno', 'fisheye'])
def test_grid_validation_accepts_every_pupil_kind_without_a_gpu(name):
    """rt_grid_create: the argument checks come before the first CUDA call -- spatial, angular and
    wide-angle grid descriptions get past them (then RT_ERR_CUDA without a device), a bad pupil kind or a
    paired list with ny != 1 is refused (RT_ERR_INVALID)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip('needs a machine WITHOUT a CUDA device')
    lib = _abi.load_library()
    spec = E.grid_spec_for_model(load_model(name), 8)
    assert spec.pupil_kind == {'dblgauss': 0, 'relay_na': 1, 'relay_fno': 2, 'fisheye': 3}[name]
    h = C.c_void_p()
    c = spec.c_spec()
    assert lib.rt_grid_create(C.byref(c), 0, C.byref(h)) == -2, lib.rt_last_error()
    c.pupil_kind = 4
    assert lib.rt_grid_create(C.byref(c), 0, C.byref(h)) == -1
    c = spec.c_spec()
    c.paired = 1
    assert lib.rt_grid_create(C.byref(c), 0, C.byref(h)) == -1


def oracle_path_tracer(path, pt0, dir0, wvl, **kw):
    """trace_raw_fn= seam: a ray over an explicit path list by the oracle"""
    from oracle import rt_oracle
    from rayoptics_b200 import raytrace as RT, trace as TR
    segs = list(path)
    descs, ns = T.describe_path(segs)
    r = rt_oracle.trace_ray(descs, ns, np.array(pt0, dtype=float), np.array(dir0, dtype=float),
                            _abi.make_opts(**{k: v for k, v in kw.items() if k in TR._TRACE_RAW_KEYS}))
    full = np.full((len(descs), 10), np.nan)
    full[:r['n_seg']] = r['ray']
    pkg, err = RT.package_ray(segs, full, r['op'], r['status'], r['fail_surf'], r['n_seg'], wvl)
    if err is not None:
        raise err
    return pkg


def test_every_bundled_lens_file_loads_and_traces(oracle):
    """All .roa / .seq / .zmx files that ship with the reference (70) go through the readers, the table
    compiler and an axial ray by the oracle.  Catalog glasses outside glass_table.json become the
    reference importers' own last resort, ConstantIndex(1.5, 'not <name>') (seq/medium.py:199-203),
    through seq.SubstituteGlasses; the one refusal is Zemax's QED surface type (which the
    reference reads as a plain sphere, zmxread.py:295-362)."""
    import glob
    import warnings
    from rayoptics_b200 import roa, seq, zmx
    root = lens_files()
    files = sorted(set(f for ext in ('roa', 'seq', 'zmx', 'ZMX')
                       for f in glob.glob(f'{root}/**/*.{ext}', recursive=True)))
    assert len(files) >= 70
    refused, substituted = [], set()
    for f in files:
        gm = seq.SubstituteGlasses()
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                opm = (roa.open_roa(f) if f.endswith('.roa') else
                       seq.open_seq(f, glass_map=gm) if f.endswith('.seq') else zmx.open_zmx(f, glass_map=gm))
        except NotImplementedError as e:
            refused.append((os.path.basename(f), str(e)))
            continue
        substituted.update(gm.not_found)
        sm, osp = opm.seq_model, opm.optical_spec
        osp._trace_raw_fn = oracle_path_tracer          # real-image-height fields trace a reverse chief ray
        descs, n_by_wvl, wvls = T.describe_model(sm)
        wide = bool(osp.field_of_view.is_wide_angle)
        pt0, dir0 = osp.ray_start_from_osp(np.array([0., 0.]), osp.field_of_view.fields[0], 'rel pupil')
        if not wide and dir0[2]*sm.z_dir[0] < 0:
            dir0 = -dir0
        r = oracle.trace_ray(descs, n_by_wvl[sm.index_for_wavelength(sm.central_wavelength())], pt0, dir0,
                             _abi.make_opts(first_surf=1, last_surf=len(descs) - 2, intersect_obj=not wide))
        assert r['status'] == 0 and r['n_seg'] == len(descs), f
        for m in (g.medium for g in sm.gaps):
            if getattr(m, 'label', '').startswith('not '):
                assert m.rindex(550.0) == 1.5
    assert [r[0] for r in refused] == ['ASL5040-UV-Zemax(ZMX).zmx'] and 'QED' in refused[0][1]
    assert 10 < len(substituted) < 60 and 'N-BK7' not in substituted
    # without the substitution policy an unknown catalog glass is an error, not a guess
    with pytest.raises(KeyError, match='glass_table'):
        seq.open_seq(f'{root}/codev/tests/ag_dblgauss.seq')


@pytest.mark.parametrize('name', ['singlet', 'dblgauss', 'triplet', 'rc', 'cellphone', 'evenasph', 'zoom52',
                                  'threemir', 'relay_na', 'telecentric'])
def test_rays_retrace_themselves_on_the_reverse_path(oracle, name):
    """Reversibility: a ray traced object -> image, turned around at the image surface and traced
    over SequentialModel.reverse_path (reverse local transforms, negated propagation directions,
    mirrors and tilted / decentered mirrors included) passes through the same point on every
    interface.  Pins reverse_path / reverse_transform against the forward machinery."""
    opm = load_model(name)
    sm, osp = opm.seq_model, opm.optical_spec
    sm.ifcs[0].interact_mode = 'dummy'
    wvl = sm.central_wavelength()
    fwd = list(sm.path(wvl))
    rev = list(sm.reverse_path(wl=wvl, start=len(sm.ifcs)))
    d_f, n_f = T.describe_path(fwd)
    d_r, n_r = T.describe_path(rev)
    n = len(fwd)
    checked = 0
    for fld in osp.field_of_view.fields:
        for pupil in ([0., 0.], [0.3, -0.5], [-0.6, 0.2]):
            pt0, dir0 = osp.ray_start_from_osp(np.array(pupil), fld, 'rel pupil')
            if dir0[2]*sm.z_dir[0] < 0:
                dir0 = -dir0
            f = oracle.trace_ray(d_f, n_f, pt0, dir0, _abi.make_opts(first_surf=1, last_surf=n - 2))
            if f['status'] != 0:
                continue
            last = f['ray'][-1]
            r = oracle.trace_ray(d_r, n_r, last[0:3], -last[3:6], _abi.make_opts(first_surf=1, last_surf=n - 2))
            assert r['status'] == 0 and r['n_seg'] == n
            for j in range(n - 1):                 # every interface but the (possibly 1e10 away) object
                p_f, p_r = f['ray'][n - 1 - j][0:3], r['ray'][j][0:3]
                assert np.abs(p_f - p_r).max() < 1e-7*max(1.0, np.abs(p_f).max()), (name, j)
            # optical path between the first and last powered surfaces is the same both ways
            assert abs(f['op'] - r['op']) < 1e-6*max(1.0, abs(f['op']))
            # the device source (general and, where the path qualifies, lean loop) on the reversed
            # path: bit-identical to the oracle
            from hostsim import build as HS
            p0 = np.ascontiguousarray(last[0:3].reshape(3, 1))
            d0 = np.ascontiguousarray(-last[3:6].reshape(3, 1))
            for kern in [0] + ([HS.lean_kind(d_r)] if HS.lean_kind(d_r) else []):
                h = HS.trace_bundle(d_r, np.array([n_r]), p0, d0, np.zeros(1, np.int32),
                                    _abi.make_opts(first_surf=1, last_surf=n - 2), kernel=kern, out_kind=2)
                assert h['status'][0] == 0 and h['op'][0] == r['op']
                assert np.array_equal(h['full'][:, :, 0], r['ray'])
            checked += 1
    assert checked >= 3
    if name == 'threemir':
        # why reverse_path does not use compute_local_transforms(step=-1) -- the restatement of the
        # reference's reverse transforms, pinned to them in test_local_transforms_equal_the_references:
        # for decentered / tilted interfaces they are not the inverses of the forward transforms
        ref_style = M.compute_local_transforms(sm.ifcs, sm.gaps, step=-1)
        worst = 0.0
        for i in range(1, n):
            rt_f, t_f = sm.lcl_tfrms[i - 1]
            rt_b, t_b = ref_style[n - 1 - i]
            assert np.array_equal(rt_b, rt_f.T)
            worst = max(worst, np.abs(t_b - (-rt_f @ t_f)).max())
        assert worst > 10.0                        # mm


def test_importers_apply_the_wide_angle_rule(tmp_path):
    """cmdproc.py:210 / zmxread.py:288: after reading, ``fov.is_wide_angle = fov.check_is_wide_angle()``
    (opticalspec.py:896-905) -- object angles beyond 45 degrees, or real image heights with the
    object at infinity -- which switches the start rays to the wide-angle construction."""
    from rayoptics_b200 import seq, zmx
    for yan, wide in ((30.0, False), (60.0, True)):
        f = tmp_path / f'w{int(yan)}.seq'
        f.write_text('\n'.join(['RDM', 'EPD 2', 'WL 587.6', f'YAN 0 {yan}', 'SO 0 1e11', 'S 20 2 517.642', ' STO',
                                'S -20 30', 'SI 0 0']))
        opm = seq.open_seq(str(f))
        fov = opm.optical_spec.field_of_view
        assert bool(fov.is_wide_angle) is wide and fov.check_is_wide_angle(optical_spec=opm.optical_spec) is wide
        recs, _, _ = opm.optical_spec.grid_fields()
        assert recs[0]['pupil_kind'] == (_abi.PUPIL_WIDE if wide else _abi.PUPIL_EPD)
    root = os.path.join(lens_files(), 'zemax', 'tests')
    kw = dict(glass_map=seq.SubstituteGlasses())
    a = zmx.open_zmx(f'{root}/US08427765-1.ZMX', **kw).optical_spec      # real heights, object at infinity
    b = zmx.open_zmx(f'{root}/US05831776-1.zmx', **kw).optical_spec      # real heights, finite object
    assert a.field_of_view.is_wide_angle and not b.field_of_view.is_wide_angle
    assert a.conjugate_type('object') == 'infinite' and b.conjugate_type('object') == 'finite'


def test_reused_grid_blocks_are_per_thread(monkeypatch):
    """analyses._reusable_grid: within a thread the device block of a grid shape is re-used
    (upload, no allocation); another thread gets its own block -- two threads running analyses on
    one device must not trace each other's grid description.  (Device grid replaced by a host
    stand-in: only the cache policy is under test.)"""
    import threading
    from rayoptics_b200 import analyses as A, engine as E

    class FakeGrid(E.PupilGridSpec):
        made = 0

        def __init__(self, *a, device=0, **k):
            super().__init__(*a, **k)
            self.device, self._handle, self.uploads = device, object(), 0
            FakeGrid.made += 1

        def upload(self, spec):
            self.uploads += 1

        def close(self):
            self._handle = None
    monkeypatch.setattr(E, 'PupilGrid', FakeGrid)
    opm = load_model('dblgauss')
    descs, n_by_wvl, wvls = T.describe_model(opm.seq_model)
    tab = type('Tab', (), {'device': 0, 'wvl_index': lambda self, w: wvls.index(w)})()
    fields, wv = list(opm.optical_spec.field_of_view.fields), list(opm.seq_model.wvlns)
    seen = {}

    def work(tag):
        g1, _ = A._reusable_grid(opm, tab, 16, fields, wv, 0.0)
        g2, _ = A._reusable_grid(opm, tab, 16, fields, wv, 0.125)      # same shape, other contents
        seen[tag] = (g1, g2, g2.uploads)
    work('main')
    t = threading.Thread(target=work, args=('other',))
    t.start()
    t.join()
    assert seen['main'][0] is seen['main'][1] and seen['main'][2] == 1
    assert seen['other'][0] is seen['other'][1] and seen['other'][0] is not seen['main'][0]
    assert FakeGrid.made == 2
