"""GPU (B200 box): the ABI v3 entry points -- reference image points computed on the device
(rt_grid_chief_ref), re-used grid blocks (rt_grid_update), NaN-coded status in the
aberration arrays (RT_OUT_ABR_NAN_STATUS), the one-launch summary combine
(rt_combine_summaries) -- and ``analyses.spot_diagram`` end to end, all against the oracle /
the earlier, separately validated entry points.  Bit-exact."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_model
from rayoptics_b200 import _abi, table as T, engine as E, analyses as A

pytestmark = pytest.mark.gpu


def np_(t):
    return t.detach().cpu().numpy()


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.fixture(scope='module')
def tables():
    cache = {}

    def get(name):
        if name not in cache:
            opm = load_model(name)
            cache[name] = (opm, T.SurfaceTable.from_model(opm.seq_model, device=0))
        return cache[name]
    return get


@pytest.mark.parametrize('name', ['dblgauss', 'rc', 'cellphone', 'exotic', 'hybrid', 'relay_na'])
def test_chief_ref_on_device_equals_the_host_round_trip(tables, name):
    """rt_grid_chief_ref writes the same reference image points that the (validated) chief-ray
    pre-pass returns to the host, for every model family (lean, poly, general, phase, angular)."""
    opm, tab = tables(name)
    sm = opm.seq_model
    fields = list(opm.optical_spec.field_of_view.fields)
    want = A.chief_ray_image_points(opm, tab, fields)                       # [n_fields, 2], host
    grid = E.grid_for_model(opm, tab, 16, ref_img=None)
    out = torch.full((len(fields), 2), float('nan'), dtype=torch.float64, device='cuda')
    grid.chief_ref(tab, tab.wvl_index(sm.central_wavelength()), out=out)
    torch.cuda.synchronize()
    assert same(np_(out), want)
    # the grid now traces with those reference points: aberrations equal a grid built from the host values
    ref_fw = np.repeat(want[:, None, :], len(sm.wvlns), axis=1)
    g2 = E.grid_for_model(opm, tab, 16, ref_img=ref_fw)
    a = E.trace_grid(tab, grid, outputs=('abr', 'status'))
    b = E.trace_grid(tab, g2, outputs=('abr', 'status'))
    torch.cuda.synchronize()
    assert same(np_(a.abr), np_(b.abr)) and same(np_(a.summary), np_(b.summary))
    grid.close(); g2.close()


def test_grid_update_reuses_the_block(tables):
    """rt_grid_update: same shape, new contents (defocus, vignetting off) == a freshly created grid;
    a different shape is refused."""
    opm, tab = tables('dblgauss')
    grid = E.grid_for_model(opm, tab, 40)
    r0 = np_(E.trace_grid(tab, grid, outputs=('abr', 'status')).abr)
    args, kw = E._grid_args(opm, tab.wvl_index, 40, None, None, 0.125, (-1.0, 1.0), False)
    grid.update(*args, **kw)
    fresh = E.PupilGrid(*args, device=0, **kw)
    a = E.trace_grid(tab, grid, outputs=('abr', 'status', 'p'))
    b = E.trace_grid(tab, fresh, outputs=('abr', 'status', 'p'))
    torch.cuda.synchronize()
    assert same(np_(a.abr), np_(b.abr)) and same(np_(a.status), np_(b.status)) and same(np_(a.p), np_(b.p))
    assert not same(np_(a.abr), r0)
    args2, kw2 = E._grid_args(opm, tab.wvl_index, 41, None, None, 0.0, (-1.0, 1.0), True)
    with pytest.raises((_abi.EngineError, ValueError)):
        grid.update(*args2, **kw2)
    fresh.close()


@pytest.mark.parametrize('name', ['dblgauss', 'cellphone', 'exotic'])
def test_nan_coded_status(tables, name):
    """RT_OUT_ABR_NAN_STATUS: finite aberrations unchanged, status / fail_surf recoverable from the NaNs."""
    opm, tab = tables(name)
    grid = E.grid_for_model(opm, tab, 48)
    plain = E.trace_grid(tab, grid, outputs=('abr', 'status', 'fail_surf'))
    coded = E.trace_grid(tab, grid, outputs=('abr',), nan_status=True)
    torch.cuda.synchronize()
    st, fs = np_(plain.status), np_(plain.fail_surf)
    assert (st != 0).any() and (st == 0).any()
    abr = np_(coded.abr)
    ok = st == 0
    assert same(abr[:, ok], np_(plain.abr)[:, ok]) and np.isnan(abr[:, ~ok]).all()
    dst, dfs = E.decode_nan_status(abr)
    assert same(dst, st) and same(dfs, fs)
    assert same(np_(coded.summary), np_(plain.summary))


def test_combine_summaries_kernel(tables):
    opm, tab = tables('dblgauss')
    grid = E.grid_for_model(opm, tab, 100)
    cuts = [0, 7, grid.n_chunks//3, grid.n_chunks - 5, grid.n_chunks]
    parts = [E.trace_grid(tab, grid, a, b, outputs=()).summary for a, b in zip(cuts[:-1], cuts[1:])]
    comb = E.combine_summaries(parts)                      # rt_combine_summaries
    torch.cuda.synchronize()
    ps = torch.stack(parts).cpu()
    want = E.combine_summaries(ps)                         # torch path on CPU tensors
    got = comb.cpu()
    assert torch.equal(got[:, 0:5], want[:, 0:5]) and torch.equal(got[:, 10:14], want[:, 10:14])
    seq = ps[0].clone()                                    # sums add in part order
    for p in ps[1:]:
        seq += p
    assert torch.equal(got[:, 5:10], seq[:, 5:10]) and torch.equal(got[:, 14], seq[:, 14])


def test_empty_chunk_range_is_the_identity(tables):
    """A rank with an empty shard contributes zeros and +-inf (min / max columns), so the combined
    summary equals the whole grid's."""
    opm, tab = tables('dblgauss')
    grid = E.grid_for_model(opm, tab, 20)
    whole = E.trace_grid(tab, grid, outputs=())
    empty = E.trace_grid(tab, grid, 3, 3, outputs=())
    torch.cuda.synchronize()
    e = np_(empty.summary)
    assert (e[:, [10, 12]] == np.inf).all() and (e[:, [11, 13]] == -np.inf).all()
    assert (np.delete(e, [10, 11, 12, 13], axis=1) == 0).all()
    comb = E.combine_summaries([whole.summary, empty.summary])
    torch.cuda.synchronize()
    assert same(np_(comb)[:, :15], np_(whole.summary)[:, :15])


def test_grid_wavelength_rows_are_range_checked(tables):
    opm, tab = tables('singlet')
    args, kw = E._grid_args(opm, tab.wvl_index, 4, None, None, 0.0, (-1.0, 1.0), True)
    bad = list(args)
    bad[1] = [tab.n_wvl + 3]
    grid = E.PupilGrid(*bad, device=0, **kw)
    with pytest.raises(_abi.EngineError, match='wvl_idx'):
        E.trace_grid(tab, grid)
    grid.close()


def spot_pieces_summary(spec, want, paths):
    """the summary spot_diagram's pieces add up to, in the documented order (test_gpu_spot_sums):
    rt_trace_grid_to_host splits the chunks at c0 + (c1 - c0)*i//n and adds the parts left to right.
    ``paths``: record path of every piece whose path the launch size leaves open."""
    from test_gpu_spot_sums import expected_summary, certain_paths, combine
    nc = spec.n_chunks
    n = min(max(1, min(8, nc//64)), nc)
    parts = []
    for i in range(n):
        cb, ce = nc*i//n, nc*(i + 1)//n
        a, b = spec.first_ray_of_chunk(cb), spec.first_ray_of_chunk(ce)
        cand = certain_paths(spec, cb, ce)
        parts.append(expected_summary(spec, cb, ce, want['abr'][:, a:b], want['op'][a:b],
                                      want['status'][a:b], cand[0] if len(cand) == 1 else paths))
    return combine(parts)


@pytest.mark.parametrize('name,num', [('dblgauss', 64), ('rc', 50), ('cellphone', 33), ('dblgauss', 512)])
def test_spot_diagram_end_to_end(tables, oracle, name, num):
    """analyses.spot_diagram (device chief rays, re-used grid block, 16 B/ray, pipelined copies):
    aberrations / status / reference points equal the oracle's, twice in a row (grid re-use); its
    statistics are spot_statistics of the summary the pieces add up to in the documented order,
    bit for bit, and lie within the rounding bound of a two-pass reference.  512^2: 8 pieces, tiles
    crossing pieces."""
    from test_gpu_spot_sums import DRYRUN, check_statistics
    opm, tab = tables(name)
    sm = opm.seq_model
    for rep in range(2):
        sd = A.spot_diagram(opm, num, table=tab)
        fields = list(opm.optical_spec.field_of_view.fields)
        ref = A.chief_ray_image_points(opm, tab, fields)
        assert same(sd.ref_img, ref)
        ref_fw = np.repeat(ref[:, None, :], len(sm.wvlns), axis=1)
        spec = E.grid_spec_for_model(opm, num, ref_img=ref_fw)
        opts = _abi.make_opts(first_surf=1, last_surf=tab.n_ifc - 2, check_apertures=True)
        want = oracle.trace_grid(spec.c_spec(), tab.descs, tab.n_by_wvl, 0, spec.n_rays, opts,
                                 n_threads=8, wvls=tab.wvls)
        ok = want['status'] == 0
        assert same(sd.status, want['status'])
        assert same(sd.fail_surf, np.where(ok, -1, want['fail_surf']))
        assert same(sd.abr[:, ok], want['abr'][:, ok])
        assert sd.io_bytes['d2h'] < 16.1*spec.n_rays + 4096
        per = num*num
        for fi in range(sd.n_fields):
            for wi in range(sd.n_wvls):
                t = fi*sd.n_wvls + wi
                m = ok[t*per:(t + 1)*per]
                assert same(sd.grids[fi][wi], want['abr'][:, t*per:(t + 1)*per][:, m].T)
                assert sd.summary['n_ok'][fi, wi] == m.sum()
        got = {k: np.asarray(v).reshape(-1) for k, v in sd.summary.items()}
        check_statistics(got, spec, want['abr'], want['op'], want['status'])
        if not DRYRUN:
            cands = [E.spot_statistics(spot_pieces_summary(spec, want, p)) for p in ('items', 'slots')]
            assert any(all(same(got[k], c[k]) for k in got) for c in cands)


@pytest.mark.parametrize('name', ['dblgauss', 'evenasph'])
def test_cuda_set_vig_batched(name):
    """vigcalc.set_vig_batched on the CUDA engine (bundles of all fields' edge searches) == the
    same searches fed by the oracle: identical vignetting factors."""
    import sys
    from rayoptics_b200 import vigcalc as V
    sys.path.insert(0, __file__.rsplit('/', 1)[0])
    from test_trace_drivers import oracle_ray_fn
    a, b = load_model(name), load_model(name)
    for m in (a, b):
        for f in m.optical_spec.field_of_view.fields:
            f.vux = f.vlx = f.vuy = f.vly = 0.0
    V.set_vig_batched(a, oracle_ray_fn(a))
    launches = V.set_vig_batched(b)                      # cuda_ray_fn
    for x, y in zip(a.optical_spec.field_of_view.fields, b.optical_spec.field_of_view.fields):
        assert (x.vux, x.vlx, x.vuy, x.vly) == (y.vux, y.vlx, y.vuy, y.vly)
    assert 0 < launches < 200
