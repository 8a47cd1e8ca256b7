"""Randomised three-way check: REFERENCE trace_raw (stored by tests/refdata.py) == oracle ==
the device source compiled for the host (tests/hostsim), bit for bit, on random systems --
random mixtures of spherical / conic / even-polynomial / radial-polynomial / toroidal profiles,
transmit / reflect / dummy / phantom interfaces, tilted and decentered transforms in both
numpy memory layouts, circular / rectangular apertures and obscurations, random trace_raw
keyword arguments (first_surf, last_surf, eps, check_apertures, intersect_obj,
filter_out_phantoms, pt_inside_fuzz) and random rays.  Seeds are fixed: failures reproduce.
"""
import numpy as np
import pytest

from rayoptics_b200 import _abi, model as M, table as T
from hostsim import build as HS
from oracle import ref_harness as rh
from refdata import digest, ref  # noqa: F401


def random_system(rng, lean=0):
    """lean: 0 anything (general kernel), 1 quadrics only / 2 quadrics + polynomials, without
    tilts and aperture lists (the lean kernels' domain)"""
    n_mid = int(rng.integers(2, 8))
    segs = []
    n_air = 1.0
    n_cur, z = n_air, 1
    n_ifc = n_mid + 2

    def rot(ax, ay):
        cx, sx, cy, sy = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay)
        return np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])

    for i in range(n_ifc):
        kind = rng.integers(0, {0: 8, 1: 4, 2: 8}[lean]) if 0 < i < n_ifc - 1 else 0
        cv = float(rng.uniform(-0.03, 0.03)) if rng.random() < 0.8 else 0.0
        if kind <= 2:
            prf = M.Spherical(cv)
        elif kind == 3:
            prf = M.Conic(c=cv, cc=float(rng.uniform(-2, 1)))
        elif kind == 4:
            prf = M.EvenPolynomial(c=cv, cc=float(rng.uniform(-1, 0.5)),
                                   coefs=[0.0, float(rng.uniform(-2e-6, 2e-6)), float(rng.uniform(-1e-9, 1e-9))])
        elif kind == 5:
            prf = M.RadialPolynomial(c=cv, ec=float(rng.uniform(0.2, 1.5)),
                                     coefs=[0.0, 0.0, float(rng.uniform(-2e-5, 2e-5)), float(rng.uniform(-1e-6, 1e-6))])
        elif kind == 6:
            prf = M.YToroid(c=cv, cR=float(rng.uniform(-0.02, 0.02)), cc=float(rng.uniform(-0.5, 0.5)),
                            coefs=[0.0, float(rng.uniform(-1e-7, 1e-7))])
        else:
            prf = M.XToroid(c=cv, cR=float(rng.uniform(-0.02, 0.02)), cc=float(rng.uniform(-0.5, 0.5)),
                            coefs=[0.0, float(rng.uniform(-1e-7, 1e-7))])
        u = rng.random()
        mode = 'dummy' if i in (0, n_ifc - 1) else ('transmit' if u < 0.6 else 'reflect' if u < 0.75
                                                    else 'dummy' if u < 0.88 else 'phantom')
        ifc = M.Surface(profile=prf, interact_mode=mode, max_aperture=float(rng.uniform(6, 14)))
        if lean == 0 and 0 < i < n_ifc - 1 and rng.random() < 0.3:
            ifc.clear_apertures = [M.Rectangular(float(rng.uniform(5, 12)), float(rng.uniform(5, 12)),
                                                 x_offset=float(rng.uniform(-1, 1)),
                                                 y_offset=float(rng.uniform(-1, 1)))]
            if rng.random() < 0.5:
                ifc.clear_apertures.append(M.Circular(float(rng.uniform(0.5, 2)), is_obscuration=True))
        if mode == 'reflect':
            z = -z
        elif mode == 'transmit':
            n_cur = n_air if (n_cur != n_air and rng.random() < 0.7) else float(rng.uniform(1.4, 1.9))
        thi = float(rng.uniform(2, 15))*z if i > 0 else float(rng.uniform(20, 60))
        if i == n_ifc - 1:
            tf = (np.identity(3), np.zeros(3))
        elif lean == 0 and rng.random() < 0.3:
            R = rot(float(rng.uniform(-0.03, 0.03)), float(rng.uniform(-0.03, 0.03)))
            R = R.T if rng.random() < 0.5 else np.ascontiguousarray(R)
            tf = (R, np.array([float(rng.uniform(-0.2, 0.2)), float(rng.uniform(-0.2, 0.2)), thi]))
        else:
            tf = (np.identity(3), np.array([0., 0., thi]))
        segs.append([ifc, None, tf, n_cur, z])
    return segs


def random_case(rng, n_ifc):
    first = int(rng.integers(0, 3))
    last = None if rng.random() < 0.2 else int(rng.integers(max(first, 1), n_ifc))
    return dict(first_surf=first, last_surf=last, check_apertures=bool(rng.random() < 0.6),
                intersect_obj=bool(rng.random() < 0.8), filter_out_phantoms=bool(rng.random() < 0.4),
                eps=float(10.0**rng.uniform(-13, -9)),
                pt_inside_fuzz=None if rng.random() < 0.6 else float(10.0**rng.uniform(-6, -2)))


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def reference_rays(segs, p0, d0, wvl, case, ks):
    """rays ks by the reference's trace_raw: [5] where it raised an uncaught error, else
    [status, n_seg, op, segments, failing surface (None if the ray got through)]"""
    path = rh.ref_path(type('S', (), {'path': lambda self, w: segs})(), wvl)
    out = []
    for k in ks:
        rr = rh.ref_trace(path, p0[:, k], d0[:, k], wvl, **case)
        out.append([5] if rr['status'] == 5 else
                   [rr['status'], rr['n_seg'], rr['op'], rr['ray'], rr['fail_surf'] if rr['status'] else None])
    return out


def oracle_rays(r, ks):
    """the same records from an oracle trace_bundle(want_full=True) result"""
    out = []
    for k in ks:
        st, n_seg = int(r['status'][k]), int(r['n_seg'][k])
        out.append([5] if st == 5 else
                   [st, n_seg, r['op'][k], r['full'][:n_seg, :, k], int(r['fail_surf'][k]) if st else None])
    return out


@pytest.mark.parametrize('lean', [0, 1, 2])
@pytest.mark.parametrize('seed', range(100))
def test_random_system_three_way(oracle, seed, lean, ref):
    rng = np.random.default_rng(1000 + seed + 100000*lean)
    segs = random_system(rng, lean)
    descs, ns = T.describe_path(segs)
    n_ifc = len(descs)
    n_by_wvl = np.array([ns])
    n = 400
    p0 = np.zeros((3, n))
    p0[:2] = rng.uniform(-6, 6, (2, n))
    tgt = rng.uniform(-5, 5, (2, n))*np.where(rng.random(n) < 0.85, 1.0, 4.0)
    v = np.array([tgt[0] - p0[0], tgt[1] - p0[1], np.full(n, abs(segs[0][2][1][2]))])
    d0 = v/np.sqrt((v*v).sum(0))
    wv = np.zeros(n, dtype=np.int32)
    case = random_case(rng, n_ifc)
    opts = _abi.make_opts(**case)
    orc = oracle.trace_bundle(descs, n_by_wvl, p0, d0, wv, opts, want_full=True, n_threads=2)
    kinds = [0] + ([HS.lean_kind(descs)] if HS.lean_kind(descs) else [])
    assert lean == 0 or len(kinds) == 2
    for kern in kinds:
        r = HS.trace_bundle(descs, n_by_wvl, p0, d0, wv, opts, kernel=kern, out_kind=2)
        for k in ('status', 'fail_surf', 'n_seg', 'op', 'last', 'full'):
            assert same(r[k], orc[k]), (seed, kern, k, case)
        if kern:                                       # the lean kernels' other output kinds
            for out_kind in (0, 1):
                r = HS.trace_bundle(descs, n_by_wvl, p0, d0, wv, opts, kernel=kern, out_kind=out_kind)
                assert same(r['status'], orc['status']) and same(r['op'], orc['op'])
                assert same(r['last'][0:6], orc['last'][0:6]) and same(r['n_seg'], orc['n_seg'])
                if out_kind == 1:
                    assert same(r['last'][6:10], orc['last'][6:10])
    # every 5th ray by the reference: status 5 where it crashed (uncaught error), else status,
    # segments, optical path and failing surface -- compared as digest()
    ks = range(0, n, 5)
    assert ref.digest(lambda: reference_rays(segs, p0, d0, 550.0, case, ks)) == digest(oracle_rays(orc, ks))


def add_phase_elements(rng, segs):
    """give some refracting / reflecting interfaces a grating, a radial DOE or a hologram"""
    for seg in segs[1:-1]:
        ifc = seg[0]
        if ifc.interact_mode not in ('transmit', 'reflect') or rng.random() < 0.5:
            continue
        u = rng.random()
        if u < 0.4:
            ifc.phase_element = M.DiffractionGrating(
                order=int(rng.choice([-1, 1, 2])), grating_lpmm=float(rng.uniform(50, 400)),
                grating_normal=[float(rng.uniform(-0.3, 0.3)), 1.0, float(rng.uniform(-0.1, 0.1))],
                interact_mode=ifc.interact_mode)
        elif u < 0.8 and ifc.interact_mode == 'transmit':
            ifc.phase_element = M.DiffractiveElement(
                coefficients=[float(rng.uniform(-2e-3, 2e-3)), float(rng.uniform(-2e-6, 2e-6)),
                              float(rng.uniform(-1e-9, 1e-9))][:int(rng.integers(1, 4))],
                ref_wl=float(rng.uniform(450, 650)), order=int(rng.choice([-1, 1, 2])))
        elif ifc.interact_mode == 'transmit':
            ifc.phase_element = M.HolographicElement(
                ref_pt=[float(rng.uniform(-5, 5)), float(rng.uniform(-5, 5)), float(rng.uniform(-200, -50))],
                ref_virtual=bool(rng.random() < 0.5),
                obj_pt=[float(rng.uniform(-5, 5)), float(rng.uniform(-5, 5)), float(rng.uniform(50, 200))],
                obj_virtual=bool(rng.random() < 0.5), ref_wl=float(rng.uniform(450, 650)))


@pytest.mark.parametrize('seed', range(60))
def test_random_phase_systems_three_way(oracle, seed, ref):
    """the same with diffractive phase elements: reference == oracle bit for bit (same libm);
    device source == oracle in status / failing surface / segment counts, coordinates within
    1e-11 mm (x**k: DESIGN.md 2a)"""
    rng = np.random.default_rng(5000 + seed)
    segs = random_system(rng, lean=0)
    add_phase_elements(rng, segs)
    wvl = 550.0
    descs, ns = T.describe_path(segs)
    n_ifc, n_by_wvl = len(descs), np.array([ns])
    n = 300
    p0 = np.zeros((3, n))
    p0[:2] = rng.uniform(-5, 5, (2, n))
    tgt = rng.uniform(-4, 4, (2, n))
    v = np.array([tgt[0] - p0[0], tgt[1] - p0[1], np.full(n, abs(segs[0][2][1][2]))])
    d0 = v/np.sqrt((v*v).sum(0))
    wv = np.zeros(n, dtype=np.int32)
    case = random_case(rng, n_ifc)
    opts = _abi.make_opts(**case)
    orc = oracle.trace_bundle(descs, n_by_wvl, p0, d0, wv, opts, want_full=True, n_threads=2, wvls=[wvl])
    r = HS.trace_bundle(descs, n_by_wvl, p0, d0, wv, opts, kernel=0, out_kind=2, wvls=[wvl])
    for k in ('status', 'fail_surf', 'n_seg'):
        assert same(r[k], orc[k]), (seed, k, case)
    assert np.array_equal(np.isnan(r['full']), np.isnan(orc['full']))
    assert np.nanmax(np.abs(r['full'] - orc['full']), initial=0.0) <= 1e-11
    assert np.nanmax(np.abs(r['op'] - orc['op']), initial=0.0) <= 1e-8
    # every 6th ray by the reference (rays it crashed on are left out), compared as digest()
    def reference_side():
        recs = reference_rays(segs, p0, d0, wvl, case, range(0, n, 6))
        crashed = [k for k, rec in zip(range(0, n, 6), recs) if rec == [5]]
        return crashed, digest([rec[:4] for rec in recs if rec != [5]])
    crashed, want = ref(reference_side)
    assert want == digest([rec[:4] for rec in oracle_rays(orc, [k for k in range(0, n, 6) if k not in crashed])])
