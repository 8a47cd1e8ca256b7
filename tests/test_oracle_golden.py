"""CPU: pin the C oracle (oracle/rt_oracle.c) to the reference.

1. against the committed golden vectors, which were produced by the reference's
   own trace_raw (tests/golden/make_golden.py) -- bit-exact;
2. against the reference's own known-answer data for this path
   (raytr/tests/marginal_ray.py via test_sequential.py:23-77, and
   elem/tests/test_profiles.py:127-154);
3. against the reference on freshly seeded rays (its results stored by tests/refdata.py).
"""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, MODEL_NAMES, PHASE_MODEL_NAMES, load_model, load_vectors
from rayoptics_b200 import _abi, table as T, model as M
from refdata import digest, ref  # noqa: F401


def same(a, b):
    """bitwise-equal values, treating NaN == NaN and -0.0 == 0.0"""
    return np.array_equal(a, b, equal_nan=True)


def run_oracle_on_vectors(oracle, name):
    opm = load_model(name)
    v = load_vectors(name)
    descs, n_by_wvl, _ = T.describe_model(opm.seq_model)
    n = v['p0'].shape[1]
    out = dict(last=np.zeros((10, n)), op=np.zeros(n), status=np.zeros(n, np.int32),
               fail_surf=np.zeros(n, np.int32), n_seg=np.zeros(n, np.int32),
               full=np.full(v['full'].shape, np.nan))
    n_full = v['full'].shape[2]
    for ci, case in enumerate(v['cases']):
        idx = np.nonzero(v['case'] == ci)[0]
        if idx.size == 0:
            continue
        opts = _abi.make_opts(**case)
        r = oracle.trace_bundle(descs, n_by_wvl, v['p0'][:, idx], v['d0'][:, idx],
                                v['wvl_idx'][idx], opts, want_full=True, wvls=opm.seq_model.wvlns)
        out['last'][:, idx] = r['last']
        for k in ('op', 'status', 'fail_surf', 'n_seg'):
            out[k][idx] = r[k]
        sel = idx < n_full
        out['full'][:, :, idx[sel]] = r['full'][:, :, sel]
    return v, out


@pytest.mark.parametrize('name', MODEL_NAMES + PHASE_MODEL_NAMES)
def test_oracle_matches_reference_vectors(oracle, name):
    v, out = run_oracle_on_vectors(oracle, name)
    assert (v['status'] <= 4).all()          # the reference never crashed on these
    assert same(out['status'], v['status'])
    assert same(out['fail_surf'], np.where(v['status'] == 0, -1, v['fail_surf']))
    assert same(out['n_seg'], v['n_seg'])
    assert same(out['op'], v['op'])
    assert same(out['last'], v['last'])
    assert same(out['full'], v['full'])


def test_kat_marginal_ray(oracle):
    """The reference's hot-path test: raytr/tests/test_sequential.py:38-77."""
    kat = json.load(open(os.path.join(GOLDEN, 'kat.json')))
    rows = [list(r) for r in kat['ag_dblgauss']]
    rows[-2][1] += rows[-1][1]
    rows[-1][1] = 0.0
    sm = M.gen_sequence(rows, wvls=[kat['wvl']], dispersion=False)   # n = n_d exactly
    descs, ns = T.describe_path(sm.path(kat['wvl']))
    p0 = np.array([0., 0., 0.])
    v = np.array([kat['epd_half'], 0., rows[0][1]])
    d0 = v/np.linalg.norm(v)
    r = oracle.trace_ray(descs, ns, p0, d0, _abi.make_opts())
    assert r['status'] == 0 and r['n_seg'] == 13
    tol = kat['rel_tol']
    for i, (seg, truth) in enumerate(zip(r['ray'], kat['marginal_ray_f1r2'])):
        xyz, tans, dist = truth
        np.testing.assert_allclose(seg[0:3], xyz, rtol=tol*10, atol=2e-6)
        np.testing.assert_allclose([seg[3]/seg[5], seg[4]/seg[5]], tans, rtol=tol*10, atol=1e-6)
        if 1 < i < 12:
            np.testing.assert_allclose(seg[6], dist, rtol=tol)


def test_kat_profile_s1(oracle):
    """elem/tests/test_profiles.py:127-154: s = 5.866433424372758 to 1e-14."""
    kat = json.load(open(os.path.join(GOLDEN, 'kat.json')))['profile_s1']
    r1, y0 = kat['r1'], kat['y0']
    # object plane at z=0, surface 1 in the same place (thi = 0): the transfer
    # to surface 1 starts from p=[0, y0, 0] with d=[0, 0, 1]
    ifcs = [M.Surface(interact_mode='dummy'), M.Surface(profile=M.Spherical(c=1/r1)),
            M.Surface(interact_mode='dummy')]
    sm = M.SequentialModel(ifcs, [M.Gap(0.0), M.Gap(10.0)])
    descs, ns = T.describe_path(sm.path())
    r = oracle.trace_ray(descs, ns, [0., y0, 0.], [0., 0., 1.], _abi.make_opts())
    s = r['ray'][0][6]
    assert s == pytest.approx(kat['s'], rel=kat['rtol'], abs=1e-14)
    sag = r1 - np.sqrt(r1*r1 - y0*y0)
    np.testing.assert_allclose(r['ray'][1][0:3], [0., y0, sag], rtol=1e-14)
    nrm = -(np.array([0., y0, sag]) - np.array([0., 0., r1]))
    np.testing.assert_allclose(r['ray'][1][7:10], nrm/np.linalg.norm(nrm), rtol=1e-14)


@pytest.mark.parametrize('backend', ['oracle', 'device source'])
def test_kat_profile_cases(oracle, backend):
    """elem/tests/test_profiles.py:36-125 (planar / convex / concave sphere, and a spherical
    EvenPolynomial that must agree with the Spherical): rays (0,0,-1) and (0,1,-1) along +z.
    ``intersect`` is reached through a one-surface path whose object plane sits 1 in front of the
    vertex, so segment 0's ``dst`` is the reference test's ``s`` and segment 1 holds the point and
    the normal.  The truths are the test file's closed forms."""
    from math import sqrt
    from hostsim import build as HS
    r = 10.0
    sag = r - sqrt(r*r - 1.0)
    cases = [(M.Spherical(c=0.0), 1.0, 0.0, 1.0, [0., 1., 0.], [0., 0., 1.]),
             (M.Spherical(c=1/r), 1.0, 0.0, 1 + sag, [0., 1., sag], None),
             (M.EvenPolynomial(c=1/r), 1.0, 0.0, 1 + sag, [0., 1., sag], None),
             (M.Conic(c=1/r, cc=0.0), 1.0, 0.0, 1 + sag, [0., 1., sag], None),
             (M.Spherical(r=-r), 1.0, 0.0, 1 - sag, [0., 1., -sag], None)]
    for prof, s0, z0, s1, pt1, n1 in cases:
        ifcs = [M.Surface(interact_mode='dummy'), M.Surface(profile=prof, max_ap=5.0),
                M.Surface(interact_mode='dummy')]
        sm = M.SequentialModel(ifcs, [M.Gap(1.0), M.Gap(10.0)])
        descs, ns = T.describe_path(sm.path())
        p = np.array([[0., 0.], [0., 1.], [0., 0.]])
        d = np.array([[0., 0.], [0., 0.], [1., 1.]])
        wv = np.zeros(2, dtype=np.int32)
        if backend == 'oracle':
            out = oracle.trace_bundle(descs, np.array([ns]), p, d, wv, _abi.make_opts(), want_full=True)
        else:
            out = HS.trace_bundle(descs, np.array([ns]), p, d, wv, _abi.make_opts(), kernel=0, out_kind=2)
        full = out['full']                                   # [n_ifc, 10, n]
        assert (out['status'] == 0).all()
        assert full[0, 6, 0] == s0 and same(full[1, 0:3, 0], np.array([0., 0., z0]))
        assert same(full[1, 7:10, 0], np.array([0., 0., 1.]))
        assert full[0, 6, 1] == pytest.approx(s1, rel=1e-14, abs=1e-14)
        np.testing.assert_allclose(full[1, 0:3, 1], pt1, rtol=1e-14, atol=1e-15)
        cv = prof.cv
        want_n = np.array([0., 0., 1.]) if cv == 0 else None
        if want_n is None:
            c = np.array([0., 0., 1/cv])
            want_n = -(np.array(pt1) - c)*np.sign(cv)
            want_n /= np.linalg.norm(want_n)
        np.testing.assert_allclose(full[1, 7:10, 1], want_n, rtol=1e-14, atol=1e-15)


def test_oracle_live_against_reference(oracle, ref):
    """Fresh seeded rays, traced by the reference and by the oracle (the segments compared as
    digest())."""
    from oracle import ref_harness as rh

    def ref_trace(path, pt0, dir0, wvl, **kw):
        r = rh.ref_trace(path, pt0, dir0, wvl, **kw)
        return {'status': r['status'], 'n_seg': r['n_seg'], 'ray': digest(r['ray']), 'op': r['op']}
    rng = np.random.default_rng(123)
    for name in ('dblgauss', 'cellphone', 'rc'):
        opm = load_model(name)
        sm = opm.seq_model
        osp = opm.optical_spec
        n_ifc = sm.get_num_surfaces()
        kw = dict(first_surf=1, last_surf=n_ifc - 2, check_apertures=True)
        opts = _abi.make_opts(**kw)
        for wi, wvl in enumerate(sm.wvlns[:2]):
            path = rh.ref_path(sm, wvl) if ref.live else None
            descs, ns = T.describe_path(sm.path(wvl))
            for fld in osp.fov.fields[::2]:
                for _ in range(12):
                    pupil = rng.uniform(-1.1, 1.1, 2)
                    pt0, dir0 = osp.ray_start_from_osp(pupil, fld, 'rel pupil')
                    a = ref(lambda: ref_trace(path, pt0, dir0, wvl, **kw))
                    b = oracle.trace_ray(descs, ns, pt0, dir0, opts)
                    assert a['status'] == b['status']
                    assert a['n_seg'] == b['n_seg']
                    assert a['ray'] == digest(b['ray'])
                    assert a['op'] == b['op']


GRID_CONFIGS = ['singlet', 'dblgauss', 'rc', 'evenasph', 'cellphone', 'zoom52', 'fisheye', 'threemir']


@pytest.mark.parametrize('name', GRID_CONFIGS)
def test_baseline_configs_grid_of_the_reference(oracle, name):
    """The five BASELINE configurations (+ the EVENASPH lens) at reduced pupil sampling: the body
    of the reference's own trace_grid loop (tests/golden/vectors/<model>_grid.npz, generator
    make_golden_grids.py) == start rays generated + traced by the oracle, bit for bit"""
    from rayoptics_b200 import engine as E
    z = np.load(os.path.join(GOLDEN, 'vectors', name + '_grid.npz'))
    opm = load_model(name)
    descs, n_by_wvl, wvls = T.describe_model(opm.seq_model)
    spec = E.grid_spec_for_model(opm, int(z['num']))
    assert spec.n_rays == z['status'].size
    wide = opm.optical_spec.field_of_view.is_wide_angle          # trace_base, trace.py:299-300
    opts = _abi.make_opts(first_surf=1, last_surf=len(descs) - 2, check_apertures=True,
                          intersect_obj=not wide)
    r = oracle.trace_grid(spec.c_spec(), descs, n_by_wvl, 0, spec.n_rays, opts, n_threads=4)
    assert same(r['status'], z['status'])
    ok = z['status'] == 0
    assert 0 < ok.sum() < ok.size
    assert same(r['last'][0:3].T[ok], z['p'][ok]) and same(r['last'][3:6].T[ok], z['d'][ok])
    assert same(r['op'][ok], z['op'][ok])
