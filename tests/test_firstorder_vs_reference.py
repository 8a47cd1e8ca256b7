"""First-order data pinned to the reference's own code.

``rayoptics.parax.firstorder`` is importable here; its ``compute_first_order``
(parax/firstorder.py:277-479) is run on light shims of the mirror model (interfaces with
``profile_cv`` / ``optical_power`` / ``interact_mode``, gaps, signed indices, the pupil and
field specifications reduced by the reference's ``derive_parax_params`` rules) and every field
of its ``FirstOrderData`` is compared, bit for bit, with rayoptics_b200/firstorder.py -- for
all fixture models: infinite and finite conjugates, mirrors, thin lenses, object- and
image-space pupil / field specifications.  The reference's numbers are stored under
tests/golden/reference/ (tests/refdata.py).
"""
import importlib
import math

import pytest

from conftest import MODEL_NAMES, PHASE_MODEL_NAMES, ANGULAR_MODEL_NAMES, load_model
from oracle import ref_harness as rh
from refdata import ref  # noqa: F401

FIELDS = ('obj_dist', 'enp_dist', 'enp_radius', 'n_obj', 'n_img', 'exp_dist', 'exp_radius',
          'obj_na', 'img_na', 'm', 'red', 'img_dist', 'efl', 'fno', 'opt_inv', 'img_ht', 'power',
          'ffl', 'bfl', 'pp1', 'ppk', 'pp_sep', 'obj_ang', 'fl_obj', 'fl_img')


def reference_parax_data(opm):
    rh.ref()
    FO = importlib.import_module('rayoptics.parax.firstorder')
    ET = importlib.import_module('rayoptics.parax.etendue')
    sm, osp = opm.seq_model, opm.optical_spec
    wvl = sm.central_wavelength()
    n_ifc = len(sm.ifcs)
    rndx = [g.medium.rindex(wvl) for g in sm.gaps] + [sm.gaps[-1].medium.rindex(wvl)]
    z_dir = list(sm.z_dir) + [sm.z_dir[-1]]
    ifcs = []
    n_before, zb = rndx[0], z_dir[0]
    for i, ifc in enumerate(sm.ifcs):            # SequentialModel.update_model, sequential.py:612-658
        thin = type(ifc).__name__ == 'ThinLens'
        za = int(math.copysign(1, zb))
        if ifc.interact_mode == 'reflect':
            za = -za
        dn = 0.0
        if i < len(sm.gaps):
            n_after = rndx[i] if za > 0 else -rndx[i]
            dn = n_after - n_before
            n_before, zb = n_after, za
        cv = ifc.optical_power if thin else ifc.profile.cv
        ifcs.append(type('Ifc', (), dict(interact_mode=ifc.interact_mode, profile_cv=cv,
                                         optical_power=ifc.optical_power if thin else dn*cv))())
    gaps = [type('Gap', (), dict(thi=g.thi, medium=g.medium))() for g in sm.gaps]

    def path(wl=None):
        for i in range(n_ifc):
            last = i >= len(gaps)
            yield [ifcs[i], None if last else gaps[i], None, None if last else rndx[i],
                   None if last else z_dir[i]]

    S = type('SM', (), {})()
    S.ifcs, S.gaps, S.z_dir, S.path = ifcs, gaps, z_dir, path
    S.central_rndx = lambda i: rndx[i]
    S.get_num_surfaces = lambda: n_ifc

    def overall_length(os_idx=1, is_idx=-1):       # sequential.py:787-804 (a plain loop: Python
        oal = 0                                    # 3.12's sum() would compensate the floats)
        for g in gaps[os_idx:is_idx]:
            oal += g.thi
        return oal
    S.overall_length = overall_length

    class Pupil:                                   # PupilSpec.derive_parax_params, opticalspec.py:619-643
        key, value = osp.pupil.key, osp.pupil.value

        def derive_parax_params(self):
            oi, k = self.key
            if 'NA' in k:
                return oi, 'slope', ET.na2slp(self.value, n=(rndx[0] if oi == 'object' else rndx[-1]))
            if 'f/#' in k:
                return oi, 'slope', -1/(2*self.value)
            return oi, 'height', self.value/2

    class Fov:                                     # FieldSpec.derive_parax_params, :823-845
        key, value = osp.field_of_view.key, osp.field_of_view.value

        def derive_parax_params(self):
            oi, k = self.key
            v = self.value if self.value != 0 else 1.
            return (oi, 'slope', ET.ang2slp(v)) if 'angle' in k else (oi, 'height', v)

    osp_shim = {'pupil': Pupil(), 'fov': Fov()}
    model = {'seq_model': S, 'optical_spec': osp_shim, 'parax_model': None, 'analysis_results': None}
    pd = FO.compute_first_order(model, sm.stop_surface, wvl)
    return {'fod': {k: getattr(pd.fod, k) for k in FIELDS},
            'ax_ray': [list(u) for u in pd.ax_ray], 'pr_ray': [list(u) for u in pd.pr_ray]}


@pytest.mark.parametrize('name', MODEL_NAMES + PHASE_MODEL_NAMES + ANGULAR_MODEL_NAMES + ['telecentric'])
def test_first_order_data_equal_the_references(name, ref):
    opm = load_model(name)
    mine = opm.optical_spec.fod
    pd = ref(lambda: reference_parax_data(opm))
    for k in FIELDS:
        a, b = getattr(mine, k), pd['fod'][k]
        assert a == b or (a != a and b != b), (k, a, b)
    assert len(mine.ax_ray) == len(pd['ax_ray'])
    for mine_ray, ref_ray in ((mine.ax_ray, pd['ax_ray']), (mine.pr_ray, pd['pr_ray'])):
        for u, v in zip(mine_ray, ref_ray):
            assert list(u) == list(v)
    assert (mine.pr_ht0, mine.pr_slp0) == (pd['pr_ray'][0][0], pd['pr_ray'][0][1])
