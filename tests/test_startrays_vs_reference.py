"""Start-ray generation pinned to the reference's own code.

`rayoptics.raytr.opticalspec` cannot be imported here (it pulls in opticalglass), so the
SOURCE TEXT of `OpticalSpecs.ray_start_from_osp` (opticalspec.py:289-400),
`FieldSpec.obj_coords` (:990-1091) and `Field.apply_vignetting` (:1339-1353) is read from
/root/reference at test time and executed in a scratch namespace on shim objects that
expose the attributes those functions read (filled from the mirror model).  Their output
is compared bit for bit with rayoptics_b200/opticalspec.py -- which the oracle and the CUDA
start-ray kernels are in turn checked against (tests/test_host.py, tests/test_hostsim.py).
The reference's results are stored under tests/golden/reference/ (tests/refdata.py).
"""
import ast
import collections
import importlib
import math

import numpy as np
import pytest

from conftest import load_model
from oracle import ref_harness as rh
from refdata import digest, ref  # noqa: F401

ParaxData = collections.namedtuple('ParaxData', ['ax_ray', 'pr_ray', 'fod'])


def reference_methods():
    R = rh.ref()
    src = open(rh.REF_SRC + '/rayoptics/raytr/opticalspec.py').read()
    tree = ast.parse(src)
    want = {('OpticalSpecs', 'ray_start_from_osp'), ('FieldSpec', 'obj_coords'),
            ('Field', 'apply_vignetting'), ('OpticalSpecs', 'conjugate_type')}
    ns = dict(np=np, math=math, normalize=R.misc_math.normalize,
              rot_v1_into_v2=R.misc_math.rot_v1_into_v2, is_fuzzy_zero=R.misc_math.is_fuzzy_zero,
              etendue=importlib.import_module('rayoptics.parax.etendue'),
              mc=importlib.import_module('rayoptics.optical.model_constants'))
    out = {}
    for cls in tree.body:
        if isinstance(cls, ast.ClassDef):
            for fn in cls.body:
                if isinstance(fn, ast.FunctionDef) and (cls.name, fn.name) in want:
                    scope = dict(ns)
                    exec(ast.get_source_segment(src, fn), scope)
                    out[(cls.name, fn.name)] = scope[fn.name]
    assert set(out) == want
    return out


class FovShim:
    def __init__(self, osp, opm_shim, methods):
        fov = osp.field_of_view
        self.key, self.value = fov.key, fov.value
        self.is_relative, self.is_wide_angle = fov.is_relative, fov.is_wide_angle
        self.optical_spec = None
        self._obj_coords = methods[('FieldSpec', 'obj_coords')]

    def obj_coords(self, fld):
        return self._obj_coords(self, fld)


class OspShim:
    def __init__(self, opm, methods):
        osp = opm.optical_spec
        fod = osp.fod
        pr = [[fod.pr_ht0, fod.pr_slp0]]                  # pr[0][mc.ht], pr[0][mc.slp]
        self.opt_model = {'analysis_results': {'parax_data': ParaxData(None, pr, fod)}}
        self.opt_model['ar'] = self.opt_model['analysis_results']
        self._parts = {'pupil': osp.pupil, 'fov': FovShim(osp, self, methods)}
        self._parts['fov'].optical_spec = self
        self._osp = osp
        self._m = methods

    def __getitem__(self, k):
        return self._parts[k]

    def obj_img_rindex(self):
        return self._osp.obj_img_rindex()

    def conjugate_type(self, space='object'):
        return self._osp.conjugate_type(space)

    def obj_coords(self, fld):
        return self._parts['fov'].obj_coords(fld)

    def ray_start_from_osp(self, pupil, fld, pupil_type='rel pupil'):
        return self._m[('OpticalSpecs', 'ray_start_from_osp')](self, pupil, fld, pupil_type)


class FldShim:
    """what Field.apply_vignetting and the start-ray code read from a field"""
    def __init__(self, f):
        self.x, self.y = f.x, f.y
        self.vux, self.vuy, self.vlx, self.vly = f.vux, f.vuy, f.vlx, f.vly
        self.aim_info = f.aim_info


def reference_start_rays(opm, pupils):
    """per field: the reference's obj_coords, and digest() of its apply_vignetting and
    ray_start_from_osp for every pupil"""
    methods = reference_methods()
    shim = OspShim(opm, methods)
    apply_vig = methods[('Field', 'apply_vignetting')]
    out = []
    for f in opm.optical_spec.field_of_view.fields:
        fs = FldShim(f)
        p_ref, d_ref = shim.obj_coords(fs)
        rays = []
        for pupil in pupils:
            v_ref = apply_vig(fs, np.array(pupil))
            pt_ref, dir_ref = shim.ray_start_from_osp(v_ref, fs, 'rel pupil')
            rays.append((v_ref, pt_ref, dir_ref))
        out.append((p_ref, d_ref, digest(rays)))
    return out


@pytest.mark.parametrize('name', ['dblgauss', 'triplet', 'rc', 'cellphone', 'thin_triplet', 'exotic',
                                  'relay_na', 'relay_fno', 'telecentric', 'singlet', 'fisheye', 'threemir'])
def test_start_rays_equal_the_references_code(name, ref):
    opm = load_model(name)
    osp = opm.optical_spec
    rng = np.random.default_rng(4)
    pupils = [np.array(p) for p in ([0., 0.], [0., 1.], [1., 0.], [-1., 0.], [0., -1.])] + \
        [rng.uniform(-1, 1, 2) for _ in range(40)]
    want = ref(lambda: reference_start_rays(opm, pupils))
    assert len(want) == len(osp.field_of_view.fields)
    for f, (p_ref, d_ref, rays_ref) in zip(osp.field_of_view.fields, want):
        p_own, d_own = osp.obj_coords(f)
        assert np.array_equal(p_ref, p_own) and np.array_equal(d_ref, d_own)
        rays = []
        for pupil in pupils:
            v_own = f.apply_vignetting(np.array(pupil))
            pt_own, dir_own = osp.ray_start_from_osp(v_own, f, 'rel pupil')
            rays.append((v_own, pt_own, dir_own))
        assert digest(rays) == rays_ref
