"""Spot sums (``rt_trace_grid``'s ``[n_tiles, 16]`` summary) against exact references.

The summary of a tile is what the kernel adds up over its rays with status 0: the leaves ``ax``,
``ay``, ``ax*ax``, ``ay*ay``, ``ax*ay`` and ``op`` (each a rounded float64 product), taken here from
the per-ray ``abr`` / ``op`` / ``status`` outputs of the same launch.  Three checks:

1. counts (columns 0-4) and min / max (10-13) equal numpy's values; column 15 is 0;
2. every sum column lies within gamma_(n-1) * sum|leaf| of ``math.fsum`` of its leaves, the
   bound that holds for any summation order;
3. every sum column equals, bit for bit, the documented order (``expected_summary``):
   - a work item (32 rays) is summed by the pairwise tree with strides 16, 8, 4, 2, 1
     (``item_sums_store`` / ``warp_record_from_regs``), rays that do not count adding +0.0;
   - ``k_reduce_summary`` splits the tile's items into 16 parts of ceil(m/16) consecutive items;
     thread t of a part sums 0.0 + item[t] + item[t+256] + ... left to right, the 256 thread sums
     are reduced by ``sh[t] += sh[t+off]`` for off = 128 ... 1, and the 16 part results are added
     left to right;
   - a launch over whole tiles gives the same value on both record paths (chunk slots and item
     sums); a launch over part of a tile keeps the items at their tile positions on the chunk-slot
     path (m = 8 * chunks_per_tile, items outside the range skipped) and re-indexes the range's
     items from its start on the item path (m = 8 * launched chunks of the tile);
   - partial summaries combine left to right (``combine_summaries``, ``rt_trace_grid_to_host``).

``B200RT_DRYRUN=1`` runs these tests on the oracle, whose summaries are long-double sums in ray
order: the bit-exact order check (3) is skipped there, checks 1 and 2 still apply.
"""
import math
import os

import numpy as np
import pytest
import torch

from conftest import load_model
from rayoptics_b200 import _abi, engine as E, table as T

DRYRUN = os.environ.get('B200RT_DRYRUN') == '1'
CHUNK = 256              # RT_BLOCK: rays per chunk
WARPS = CHUNK//32        # work items per chunk
SPLIT = 16               # RT_RED_SPLIT: reduction parts per tile
RED_THREADS = 256        # RT_RED_THREADS
SUM_COLS = (5, 6, 7, 8, 9, 14)
MIN_COLS, MAX_COLS = (10, 12), (11, 13)
SM_COUNT_B200 = 148
U = 2.0**-53


def np_(t):
    return t.detach().cpu().numpy()


def leaves(abr, op):
    """[6, n]: the values summed into columns 5, 6, 7, 8, 9, 14"""
    ax, ay = abr[0], abr[1]
    return np.stack([ax, ay, ax*ax, ay*ay, ax*ay, op])


# ----------------------------------------------------------------- the documented order
def item_tree(v):
    """[c, m, 32] -> [c, m]: pairwise sums of each 32-ray work item, strides 16, 8, 4, 2, 1"""
    for s in (16, 8, 4, 2, 1):
        v = v[..., :s] + v[..., s:2*s]
    return v[..., 0]


def reduce_items(items):
    """[c, m] item sums in item order -> [c]: k_reduce_summary's order (16 parts, 256 threads)"""
    nc, m = items.shape
    per = -(-m//SPLIT)
    total = None
    for p in range(SPLIT):
        seg = items[:, p*per:min((p + 1)*per, m)]
        sh = np.zeros((nc, RED_THREADS))
        for j in range(0, seg.shape[1], RED_THREADS):
            blk = seg[:, j:j + RED_THREADS]
            sh[:, :blk.shape[1]] = sh[:, :blk.shape[1]] + blk
        off = RED_THREADS//2
        while off:
            sh[:, :off] = sh[:, :off] + sh[:, off:2*off]
            off //= 2
        total = sh[:, 0].copy() if total is None else total + sh[:, 0]
    return total


def identity_row():
    row = np.zeros(_abi.RT_SUMMARY_DOUBLES)
    row[list(MIN_COLS)], row[list(MAX_COLS)] = np.inf, -np.inf
    return row


def tile_rays(grid, c0, c1, t):
    """chunks [a, b) of tile t inside [c0, c1) and their rays (flattened indices), or None"""
    cpt = grid.chunks_per_tile
    a, b = max(c0, t*cpt), min(c1, (t + 1)*cpt)
    if a >= b:
        return None
    return a, b, grid.first_ray_of_chunk(a), grid.first_ray_of_chunk(b)


def expected_summary(grid, c0, c1, abr, op, status, path='items'):
    """The summary of a launch over chunks [c0, c1) as k_reduce_summary produces it, from the
    launch's per-ray outputs (arrays over the rays of [c0, c1)).  ``path``: 'items' or 'slots'
    (the same value for launches over whole tiles)."""
    cpt = grid.chunks_per_tile
    base = grid.first_ray_of_chunk(c0)
    out = np.tile(identity_row(), (grid.n_tiles, 1))
    lv_all = leaves(abr, op)
    for t in range(grid.n_tiles):
        rng = tile_rays(grid, c0, c1, t)
        if rng is None:
            continue
        a, b, r0, r1 = rng
        st = status[r0 - base:r1 - base]
        ok = st == 0
        row = out[t]
        row[0:4] = [(st == s).sum() for s in range(4)]
        row[4] = (st > 3).sum()
        lv = lv_all[:, r0 - base:r1 - base]
        if ok.any():
            row[10], row[11] = lv[0, ok].min(), lv[0, ok].max()
            row[12], row[13] = lv[1, ok].min(), lv[1, ok].max()
        pad = np.zeros((6, cpt*CHUNK))
        lo = (a - t*cpt)*CHUNK
        pad[:, lo:lo + (r1 - r0)] = np.where(ok, lv, 0.0)
        items = item_tree(pad.reshape(6, cpt*WARPS, 32))
        if path == 'items':
            items = items[:, (a - t*cpt)*WARPS:(b - t*cpt)*WARPS]
        row[list(SUM_COLS)] = reduce_items(items)
    return out


def combine(parts):
    """combine_summaries / rt_trace_grid_to_host: parts added (min / max) left to right"""
    v = parts[0].copy()
    mn, mx = list(MIN_COLS), list(MAX_COLS)
    for p in parts[1:]:
        lo, hi = np.fmin(v[:, mn], p[:, mn]), np.fmax(v[:, mx], p[:, mx])
        v = v + p
        v[:, mn], v[:, mx] = lo, hi
    return v


def certain_paths(grid, c0, c1):
    """Record paths a launch over [c0, c1) may take.  The kernel uses chunk slots when
    chunks_per_tile <= its grid size, which is at most min(launched chunks, 8 CTAs x SMs, 2048):
    fewer launched chunks than chunks_per_tile => items; chunks_per_tile <= SM count and at least
    that many launched chunks => slots; otherwise it depends on the occupancy."""
    cpt, n = grid.chunks_per_tile, c1 - c0
    if n < cpt or cpt > min(8*SM_COUNT_B200, 2048):
        return ('items',)
    if cpt <= SM_COUNT_B200:
        return ('slots',)
    return ('items', 'slots')


# ----------------------------------------------------------------- checks
def gamma(k):
    return k*U/(1 - k*U)


def check_exact_and_bound(summ, grid, c0, c1, abr, op, status):
    """checks 1 and 2 of the module docstring"""
    want = expected_summary(grid, c0, c1, abr, op, status)
    exact = [0, 1, 2, 3, 4, 10, 11, 12, 13]
    assert np.array_equal(summ[:, exact], want[:, exact])
    assert (summ[:, 15] == 0).all()
    base = grid.first_ray_of_chunk(c0)
    lv_all = leaves(abr, op)
    for t in range(grid.n_tiles):
        rng = tile_rays(grid, c0, c1, t)
        if rng is None or want[t, 0] == 0:
            assert (summ[t, list(SUM_COLS)] == 0).all() and not np.signbit(summ[t, list(SUM_COLS)]).any()
            continue
        _, _, r0, r1 = rng
        ok = status[r0 - base:r1 - base] == 0
        lv = lv_all[:, r0 - base:r1 - base][:, ok]
        n = lv.shape[1]
        for k, col in enumerate(SUM_COLS):
            ref = math.fsum(lv[k])
            bound = gamma(max(n - 1, 1))*math.fsum(np.abs(lv[k]))*(1 + 4*U) + U*abs(ref)
            assert abs(summ[t, col] - ref) <= bound, (t, col, summ[t, col], ref, bound)


def check_order(summ, grid, c0, c1, abr, op, status, paths=None):
    """check 3: bit for bit against the documented order; returns the path that matched"""
    if DRYRUN:
        return None
    paths = certain_paths(grid, c0, c1) if paths is None else paths
    for path in paths:
        want = expected_summary(grid, c0, c1, abr, op, status, path)
        if np.array_equal(summ[:, :15], want[:, :15]):
            return path
    raise AssertionError(f'summary of chunks [{c0}, {c1}) differs from the documented order '
                         f'(paths {paths})')


def check_statistics(summ, grid, abr, op, status):
    """spot_statistics of a whole-grid summary against a two-pass reference with fsum; the
    tolerance is the rounding of the one-pass formula var = (Sxx + Syy)/n - (cx^2 + cy^2).
    ``summ``: the summary, or its spot_statistics as a dict of per-tile arrays."""
    s = summ if isinstance(summ, dict) else E.spot_statistics(summ)
    rpt = grid.rays_per_tile
    for t in range(grid.n_tiles):
        sl = slice(t*rpt, (t + 1)*rpt)
        ok = status[sl] == 0
        n = int(ok.sum())
        assert s['n_ok'][t] == n
        if n == 0:
            continue
        ax, ay, o = abr[0, sl][ok], abr[1, sl][ok], op[sl][ok]
        assert s['min_x'][t] == ax.min() and s['max_x'][t] == ax.max()
        assert s['min_y'][t] == ay.min() and s['max_y'][t] == ay.max()
        g = gamma(n + 4)
        mx, my, mo = math.fsum(ax)/n, math.fsum(ay)/n, math.fsum(o)/n
        amx, amy, amo = math.fsum(np.abs(ax))/n, math.fsum(np.abs(ay))/n, math.fsum(np.abs(o))/n
        tol_cx, tol_cy = g*amx + U*abs(mx), g*amy + U*abs(my)
        assert abs(s['centroid_x'][t] - mx) <= tol_cx
        assert abs(s['centroid_y'][t] - my) <= tol_cy
        assert abs(s['mean_op'][t] - mo) <= g*amo + U*abs(mo)
        var = math.fsum((ax - mx)**2 + (ay - my)**2)/n          # two-pass reference
        m2 = math.fsum(ax*ax + ay*ay)/n
        # (Sxx + Syy)/n: gamma_(n+2) * m2; cx^2 + cy^2: 2|c| * tol_c + gamma_2 * c^2 each;
        # the final subtraction and the reference's own rounding: 4u * (m2 + var)
        err = g*m2 + 2*(abs(mx) + tol_cx)*tol_cx + 2*(abs(my) + tol_cy)*tol_cy \
            + gamma(2)*(mx*mx + my*my) + 4*U*(m2 + var)
        rms = s['rms_radius'][t]
        tol_rms = (err/math.sqrt(var) if var > 0 else math.sqrt(err)) + 2*U*rms
        assert abs(rms - math.sqrt(var)) <= tol_rms, (t, rms, math.sqrt(var), tol_rms)


def check_launch(summ, grid, c0, c1, abr, op, status, paths=None):
    check_exact_and_bound(summ, grid, c0, c1, abr, op, status)
    return check_order(summ, grid, c0, c1, abr, op, status, paths)


# ----------------------------------------------------------------- CPU: helper == literal loops
def _shfl_xor(vals, m):
    return [vals[lane ^ m] for lane in range(32)]


def _literal_item_sums_store(ok, ax, ay, op):
    """item_sums_store (b200rt.cu), lane by lane: 32 lanes -> the 6 values of lanes 4g"""
    v = [[ax[l] if ok[l] else 0.0, ay[l] if ok[l] else 0.0, ax[l]*ax[l] if ok[l] else 0.0,
          ay[l]*ay[l] if ok[l] else 0.0, ax[l]*ay[l] if ok[l] else 0.0, op[l] if ok[l] else 0.0,
          0.0, 0.0] for l in range(32)]
    h16 = [bool(l & 16) for l in range(32)]
    h8 = [bool(l & 8) for l in range(32)]
    h4 = [bool(l & 4) for l in range(32)]
    a = []
    for j in range(4):
        send = [v[l][j] if h16[l] else v[l][j + 4] for l in range(32)]
        recv = _shfl_xor(send, 16)
        a.append([(v[l][j + 4] if h16[l] else v[l][j]) + recv[l] for l in range(32)])
    b = []
    for j in range(2):
        send = [a[j][l] if h8[l] else a[j + 2][l] for l in range(32)]
        recv = _shfl_xor(send, 8)
        b.append([(a[j + 2][l] if h8[l] else a[j][l]) + recv[l] for l in range(32)])
    send = [b[0][l] if h4[l] else b[1][l] for l in range(32)]
    recv = _shfl_xor(send, 4)
    c = [(b[1][l] if h4[l] else b[0][l]) + recv[l] for l in range(32)]
    r = _shfl_xor(c, 2)
    c = [c[l] + r[l] for l in range(32)]
    r = _shfl_xor(c, 1)
    c = [c[l] + r[l] for l in range(32)]
    dst = [None]*6
    for lane in range(32):
        idx = ((lane >> 4) & 1)*4 + ((lane >> 3) & 1)*2 + ((lane >> 2) & 1)
        if (lane & 3) == 0 and idx < 6:
            dst[idx] = c[lane]
    return dst


def _literal_record_from_regs(ok, ax, ay, op):
    """warp_record_from_regs, sum columns only: shfl_down tree, lane 0's value"""
    out = []
    for k in range(6):
        x = [(ax[l], ay[l], ax[l]*ax[l], ay[l]*ay[l], ax[l]*ay[l], op[l])[k] if ok[l] else 0.0
             for l in range(32)]
        off = 16
        while off:
            y = [x[l + off] if l + off < 32 else x[l] for l in range(32)]
            x = [x[l] + y[l] for l in range(32)]
            off >>= 1
        out.append(x[0])
    return out


def _literal_launch(rpt, cpt, n_tiles, cb, ce, ax, ay, op, ok, chunk_slots):
    """grid_chunk_loop's sum records + k_reduce_summary (sum columns), loop by loop.
    ax, ay, op, ok: per-ray arrays of the whole grid (flattened tile-major)."""
    sl = min(cpt, 2048)
    recs = np.zeros((n_tiles*sl*WARPS, 16))
    n_items = (ce - cb)*WARPS
    item_sums = np.zeros((n_items, 6))
    for item in range(n_items):                 # the order items are drawn in does not matter
        c = cb + item//WARPS
        s = item % WARPS
        tile, lc = divmod(c, cpt)
        lanes_ok, lx, ly, lo = [False]*32, [0.0]*32, [0.0]*32, [0.0]*32
        for lane in range(32):
            loc = lc*CHUNK + s*32 + lane
            if loc < rpt:
                k = tile*rpt + loc
                lanes_ok[lane], lx[lane], ly[lane], lo[lane] = bool(ok[k]), ax[k], ay[k], op[k]
        if chunk_slots:
            rec = recs[(tile*sl + lc)*WARPS + s]
            for j, col in enumerate(SUM_COLS):
                rec[col] = _literal_record_from_regs(lanes_ok, lx, ly, lo)[j]
            rec[15] = 1.0
        else:
            item_sums[item] = _literal_item_sums_store(lanes_ok, lx, ly, lo)
    if not chunk_slots:                         # acc_flush records: counts only, sums 0.0
        for t in range(n_tiles):
            for r in range(sl*WARPS):
                if cb < (t + 1)*cpt and ce > t*cpt:
                    recs[t*sl*WARPS + r, 15] = 1.0
    recs_per_tile = sl*WARPS
    summary = np.zeros((n_tiles, 6))
    for tile in range(n_tiles):
        partials = []
        for part in range(SPLIT):
            per = (recs_per_tile + SPLIT - 1)//SPLIT
            r0, r1 = part*per, min(part*per + per, recs_per_tile)
            x = [[0.0]*6 for _ in range(RED_THREADS)]
            for t in range(RED_THREADS):
                r = r0 + t
                while r < r1:
                    p = recs[tile*recs_per_tile + r]
                    if p[15] != 0.0:
                        for j, col in enumerate(SUM_COLS):
                            x[t][j] = x[t][j] + p[col]
                    r += RED_THREADS
            if not chunk_slots:
                c0, c1 = max(tile*cpt, cb), min(tile*cpt + cpt, ce)
                if c1 > c0:
                    i0, n_it = (c0 - cb)*WARPS, (c1 - c0)*WARPS
                    per_it = (n_it + SPLIT - 1)//SPLIT
                    a0, a1 = part*per_it, min(part*per_it + per_it, n_it)
                    for t in range(RED_THREADS):
                        it = a0 + t
                        while it < a1:
                            for j in range(6):
                                x[t][j] += item_sums[i0 + it][j]
                            it += RED_THREADS
            off = RED_THREADS//2
            while off:
                for t in range(off):
                    x[t] = [x[t][j] + x[t + off][j] for j in range(6)]
                off >>= 1
            partials.append(x[0])
        v = partials[0]
        for p in partials[1:]:
            v = [v[j] + p[j] for j in range(6)]
        summary[tile] = v
    return summary


class _Dims:
    def __init__(self, rpt, n_tiles):
        self.rays_per_tile, self.n_tiles = rpt, n_tiles
        self.chunks_per_tile = -(-rpt//CHUNK)
        self.n_chunks = n_tiles*self.chunks_per_tile
    first_ray_of_chunk = E.PupilGridSpec.first_ray_of_chunk
    chunk_rays = CHUNK


@pytest.mark.parametrize('seed', range(6))
def test_order_helper_matches_the_kernel_loops(seed):
    """expected_summary == a literal transcription of item_sums_store / warp_record_from_regs +
    k_reduce_summary, on small random tiles, whole and partial launches, both record paths"""
    rng = np.random.default_rng(seed)
    rpt = int(rng.choice([1, 31, 257, 1000, 4099, 9000, 17000]))
    n_tiles = int(rng.integers(1, 4))
    g = _Dims(rpt, n_tiles)
    n = rpt*n_tiles
    scale = 10.0**rng.uniform(-6, 6, (3, n))         # wide dynamic range: the order shows
    ax, ay, op = (rng.standard_normal((3, n))*scale)
    ok = rng.random(n) < 0.8
    status = np.where(ok, 0, rng.integers(1, 6, n)).astype(np.int32)
    ranges = [(0, g.n_chunks)]
    for _ in range(2):
        a = int(rng.integers(0, g.n_chunks))
        ranges.append((a, int(rng.integers(a + 1, g.n_chunks + 1))))
    for cb, ce in ranges:
        r0, r1 = g.first_ray_of_chunk(cb), g.first_ray_of_chunk(ce)
        abr = np.stack([ax[r0:r1], ay[r0:r1]])
        for path in ('items', 'slots'):
            lit = _literal_launch(rpt, g.chunks_per_tile, n_tiles, cb, ce, ax, ay, op, ok,
                                  path == 'slots')
            got = expected_summary(g, cb, ce, abr, op[r0:r1], status[r0:r1], path)
            assert np.array_equal(got[:, list(SUM_COLS)], lit), (cb, ce, path)
        if cb % g.chunks_per_tile == 0 and ce % g.chunks_per_tile == 0:
            a = expected_summary(g, cb, ce, abr, op[r0:r1], status[r0:r1], 'items')
            b = expected_summary(g, cb, ce, abr, op[r0:r1], status[r0:r1], 'slots')
            assert np.array_equal(a, b)


def test_combine_left_to_right():
    rng = np.random.default_rng(5)
    parts = [rng.standard_normal((3, 16))*10.0**rng.uniform(-8, 8, (3, 16)) for _ in range(5)]
    got = combine(parts)
    for t in range(3):
        for k in range(16):
            v = parts[0][t, k]
            for p in parts[1:]:
                v = min(v, p[t, k]) if k in MIN_COLS else max(v, p[t, k]) if k in MAX_COLS else v + p[t, k]
            assert got[t, k] == v


# ----------------------------------------------------------------- GPU
@pytest.fixture(scope='module')
def tables():
    cache = {}

    def get(name):
        if name not in cache:
            opm = load_model(name)
            cache[name] = (opm, T.SurfaceTable.from_model(opm.seq_model, device=0))
        return cache[name]
    return get


def sample_against_oracle(oracle, tab, grid, c0, c1, abr, op, status, n=6, seed=0):
    """a seeded sample of the launch's chunks against the oracle"""
    rng = np.random.default_rng(seed)
    opts = _abi.make_opts(first_surf=1, last_surf=tab.n_ifc - 2, check_apertures=True)
    base = grid.first_ray_of_chunk(c0)
    for c in rng.integers(c0, c1, n):
        a, b = grid.first_ray_of_chunk(int(c)), grid.first_ray_of_chunk(int(c) + 1)
        ref = oracle.trace_grid(grid.c_spec(), tab.descs, tab.n_by_wvl, a, b, opts, n_threads=8,
                                wvls=tab.wvls)
        sl = slice(a - base, b - base)
        assert np.array_equal(status[sl], ref['status'])
        assert np.array_equal(op[sl], ref['op'], equal_nan=True)
        assert np.array_equal(abr[:, sl], ref['abr'], equal_nan=True)


def run_and_check(oracle, tab, grid, c0=0, c1=None, paths=None):
    c1 = grid.n_chunks if c1 is None else c1
    r = E.trace_grid(tab, grid, c0, c1, outputs=('abr', 'op', 'status'))
    torch.cuda.synchronize()
    abr, op, st, summ = np_(r.abr), np_(r.op), np_(r.status), np_(r.summary)
    sample_against_oracle(oracle, tab, grid, c0, c1, abr, op, st)
    path = check_launch(summ, grid, c0, c1, abr, op, st, paths)
    return r, path


@pytest.mark.gpu
@pytest.mark.parametrize('name,num,path', [
    ('dblgauss', 100, 'slots'),        # 40 chunks per tile
    ('dblgauss', 600, 'items'),        # 1407 chunks per tile > 8 CTAs x 148 SMs
    ('rc', 1024, 'items'),             # 4096 chunks per tile: record slots capped at 2048
    ('cellphone', 33, 'slots'),        # 5 chunks per tile, the last item partial; polynomial lean
    ('exotic', 33, 'slots'),           # general kernels
])
def test_whole_grid_sums(tables, oracle, name, num, path):
    opm, tab = tables(name)
    grid = E.grid_for_model(opm, tab, num)
    if not DRYRUN:
        assert certain_paths(grid, 0, grid.n_chunks) == (path,)
    r, _ = run_and_check(oracle, tab, grid)
    st = np_(r.status)
    assert (st == 0).mean() > 0.3 and (st != 0).any()
    check_statistics(np_(r.summary), grid, np_(r.abr), np_(r.op), st)


@pytest.mark.gpu
def test_paired_list_grid_sums(tables, oracle):
    """a list of 1000 pupil points per field (paired: ny = 1), 4 chunks per tile"""
    opm, tab = tables('dblgauss')
    args, kw = E._grid_args(opm, tab.wvl_index, 2, None, None, None, (-1.0, 1.0), True)
    rng = np.random.default_rng(2)
    nf = len(args[0])
    px, py = rng.uniform(-1.05, 1.05, (2, nf, 1000))
    grid = E.PupilGrid(args[0], args[1], px, py, *args[4:], paired=True, device=0, **kw)
    assert (grid.nx, grid.ny, grid.chunks_per_tile) == (1000, 1, 4)
    r, _ = run_and_check(oracle, tab, grid)
    check_statistics(np_(r.summary), grid, np_(r.abr), np_(r.op), np_(r.status))


@pytest.mark.gpu
def test_no_ray_through_gives_identities(tables, oracle):
    """a pupil range wholly outside the aperture: every count but the blocked ones is 0, the
    sums are +0.0, min = +inf and max = -inf"""
    opm, tab = tables('dblgauss')
    grid = E.grid_for_model(opm, tab, 40, pupil_range=(3.0, 4.0))
    r, _ = run_and_check(oracle, tab, grid)
    summ = np_(r.summary)
    assert (summ[:, 0] == 0).all() and (summ[:, 1:5].sum(1) == grid.rays_per_tile).all()
    assert (summ[:, list(SUM_COLS)] == 0).all() and not np.signbit(summ[:, list(SUM_COLS)]).any()
    assert (summ[:, list(MIN_COLS)] == np.inf).all() and (summ[:, list(MAX_COLS)] == -np.inf).all()


@pytest.mark.gpu
@pytest.mark.parametrize('num', [100, 600])
def test_shards_and_their_combination(tables, oracle, num):
    """chunk ranges that cross tile boundaries, on both record paths, and combine_summaries of
    them (left to right) -- which also equals tracing the pieces through rt_trace_grid_to_host"""
    opm, tab = tables('dblgauss')
    grid = E.grid_for_model(opm, tab, num)
    cpt, nc = grid.chunks_per_tile, grid.n_chunks
    cuts = [0, 7, cpt - 3, cpt + 5, 2*cpt + cpt//2, 5*cpt + 1, nc]
    parts, seen = [], set()
    for a, b in zip(cuts[:-1], cuts[1:]):
        r, path = run_and_check(oracle, tab, grid, a, b)
        parts.append(np_(r.summary))
        seen.add(path)
    if not DRYRUN and num == 100:
        assert seen == {'items', 'slots'}
    comb = E.combine_summaries([torch.as_tensor(p, device='cuda') for p in parts])
    torch.cuda.synchronize()
    comb = np_(comb)
    whole = E.trace_grid(tab, grid, outputs=('abr', 'op', 'status'))
    torch.cuda.synchronize()
    abr, op, st = np_(whole.abr), np_(whole.op), np_(whole.status)
    check_exact_and_bound(comb, grid, 0, nc, abr, op, st)
    if not DRYRUN:
        assert np.array_equal(comb, combine(parts))
    check_statistics(comb, grid, abr, op, st)
