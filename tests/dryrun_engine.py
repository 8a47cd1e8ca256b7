"""Dry-run engine for the GPU test files (TEST INFRASTRUCTURE, opt-in, never used by the driver).

    B200RT_DRYRUN=1 python -m pytest tests/test_zz_gpu_additions.py -m gpu -q

replaces the CUDA entry points of rayoptics_b200.engine / table with stand-ins that compute the
same results with the oracle on CPU tensors, so that GPU test CODE written without access to a
GPU (API use, shapes, tolerances, fixtures) can be exercised before it first meets the hardware.
It says nothing about the kernels -- that is what the real `-m gpu` run is for.
"""
import numpy as np
import torch

from oracle import rt_oracle
from rayoptics_b200 import _abi, engine as E, table as T, analyses as A


class DryTable:
    def __init__(self, descs, n_by_wvl, wvls=None, device=0):
        self.descs, self.n_by_wvl = descs, np.ascontiguousarray(n_by_wvl, dtype=np.float64)
        self.n_ifc, self.n_wvl = len(descs), self.n_by_wvl.shape[0]
        self.wvls = list(wvls) if wvls is not None else list(range(self.n_wvl))
        self.device, self.handle = int(device), object()
        self._handle = self.handle

    def wvl_index(self, wvl):
        return self.wvls.index(wvl)

    def close(self):
        pass


def _from_model(cls, seq_model, device=0, wvls=None):
    descs, n_by_wvl, wv = T.describe_model(seq_model, wvls)
    return DryTable(descs, n_by_wvl, wv, device)


def _from_path(cls, path, device=0, wvl=None):
    descs, ns = T.describe_path(path)
    return DryTable(descs, np.array([ns]), None if wvl is None else [float(wvl)], device)


class DryGrid(E.PupilGridSpec):
    def __init__(self, *args, device=0, **kwargs):
        super().__init__(*args, **kwargs)
        self.device, self.handle = int(device), object()
        self._handle = self.handle

    def host_bytes(self):
        return 0

    def close(self):
        pass

    def shape_key(self):
        return (self.device, self.n_fields, self.n_wvls, self.nx, self.ny, self.paired,
                self.wave is not None)

    def update(self, *args, **kwargs):
        kwargs.pop('device', None)
        old = self.shape_key()
        E.PupilGridSpec.__init__(self, *args, **kwargs)
        if self.shape_key() != old:
            raise ValueError('PupilGrid.update: the new description has a different shape')
        return self

    def upload(self, spec):
        keep = (self.device, self.handle)
        self.__dict__.update(spec.__dict__)
        self.device, self.handle = keep
        return self

    def chief_ref(self, table, wvl_idx, out=None):
        """rt_grid_chief_ref: chief rays (pupil 0,0, apertures not checked) of every field at
        index row ``wvl_idx``; their image intercepts become the reference points of all tiles"""
        spec = object.__new__(E.PupilGridSpec)           # same fields, one (0, 0) pupil point
        spec.__dict__.update(self.__dict__)
        nf = self.n_fields
        spec.pupil_x = spec.pupil_y = np.zeros((nf, 1))
        spec.nx = spec.ny = spec.rays_per_tile = spec.chunks_per_tile = 1
        spec.wvl_idx, spec.n_wvls = np.array([int(wvl_idx)], dtype=np.int32), 1
        spec.ref_img = spec.wave = None
        spec.apply_vignetting, spec.paired = 1, 0
        spec.n_tiles = spec.n_chunks = spec.n_rays = nf
        opts = dict(first_surf=1, last_surf=table.n_ifc - 2, check_apertures=False)
        if self.pupil_kind == _abi.PUPIL_WIDE:
            opts['intersect_obj'] = False
        g = rt_oracle.trace_grid(spec.c_spec(), table.descs, table.n_by_wvl, 0, spec.n_rays,
                                 _abi.make_opts(**opts), wvls=table.wvls)
        ref = g['last'][0:2].T.copy()                                    # [n_fields, 2]
        self.ref_img = np.repeat(ref[:, None, :], self.n_wvls, axis=1)
        if out is not None:
            out.copy_(torch.from_numpy(ref))
        return out


def _result(n, n_ifc, outputs, full):
    return E.BundleResult(n, n_ifc, torch.device('cpu'), tuple(outputs) + (('full',) if full else ()))


def _fill(res, r, keys):
    t = torch.from_numpy
    if res.p is not None:
        res.p.copy_(t(r['last'][0:3].copy()))
    if res.d is not None:
        res.d.copy_(t(r['last'][3:6].copy()))
    if res.dst is not None:
        res.dst.copy_(t(r['last'][6].copy()))
    if res.nrml is not None:
        res.nrml.copy_(t(r['last'][7:10].copy()))
    for k in ('op', 'status', 'fail_surf', 'n_seg'):
        if getattr(res, k) is not None and k in r:
            getattr(res, k).copy_(t(np.ascontiguousarray(r[k])))
    if res.full is not None:
        res.full.copy_(t(r['full']))


def trace_bundle(table, p, d, wvl_idx=None, full=False, outputs=E.BUNDLE_OUTPUTS, **kwargs):
    p = np.ascontiguousarray(torch.as_tensor(p).cpu().numpy(), dtype=np.float64).reshape(3, -1)
    d = np.ascontiguousarray(torch.as_tensor(d).cpu().numpy(), dtype=np.float64).reshape(3, -1)
    n = p.shape[1]
    wi = table.wvl_index(kwargs.pop('wvl')) if 'wvl' in kwargs else 0
    wi = kwargs.pop('wvl_index', wi)
    wv = np.full(n, wi, np.int32) if wvl_idx is None else np.asarray(torch.as_tensor(wvl_idx).cpu().numpy(), np.int32)
    r = rt_oracle.trace_bundle(table.descs, table.n_by_wvl, p, d, wv, _abi.make_opts(**kwargs),
                               want_full=True, n_threads=4, wvls=table.wvls)
    res = _result(n, table.n_ifc, outputs, full)
    _fill(res, r, outputs)
    return res


def trace_grid(table, grid, chunk_begin=0, chunk_end=None, outputs=E.GRID_OUTPUTS, full=False,
               summary=True, res=None, nan_status=False, **kwargs):
    chunk_end = grid.n_chunks if chunk_end is None else chunk_end
    kwargs.setdefault('check_apertures', True)
    kwargs.setdefault('first_surf', 1)
    kwargs.setdefault('last_surf', table.n_ifc - 2)
    if grid.pupil_kind == _abi.PUPIL_WIDE:
        kwargs['intersect_obj'] = False
    if (np.asarray(grid.wvl_idx) >= table.n_wvl).any() or (np.asarray(grid.wvl_idx) < 0).any():
        raise _abi.EngineError('rt_trace_grid: wvl_idx out of range for this table')
    opts = _abi.make_opts(**kwargs)
    r0, r1 = grid.first_ray_of_chunk(chunk_begin), grid.first_ray_of_chunk(chunk_end)
    spec = grid.c_spec()
    g = rt_oracle.trace_grid(spec, table.descs, table.n_by_wvl, r0, r1, opts, n_threads=4, wvls=table.wvls)
    if full or 'n_seg' in outputs or (res is not None and (res.full is not None or res.n_seg is not None)):
        p, d, wv, _ = rt_oracle.grid_start_rays(spec, r0, r1)
        b = rt_oracle.trace_bundle(table.descs, table.n_by_wvl, p, d, wv, opts, want_full=True,
                                   n_threads=4, wvls=table.wvls)
        g['full'], g['n_seg'] = b['full'], b['n_seg']
    if res is None:
        res = _result(r1 - r0, table.n_ifc, outputs, full)
        res.nan_status = bool(nan_status)
    _fill(res, g, outputs)
    if res.abr is not None:
        abr = g['abr'].copy()
        if nan_status:
            bad = g['status'] != 0
            bits = abr.view(np.uint64)
            bits[0, bad] = _abi.RT_NAN_PAYLOAD_BASE | g['status'][bad].astype(np.uint64)
            bits[1, bad] = _abi.RT_NAN_PAYLOAD_BASE | g['fail_surf'][bad].astype(np.uint64)
        res.abr.copy_(torch.from_numpy(abr))
    if res.opd is not None and g['opd'] is not None:
        res.opd.copy_(torch.from_numpy(g['opd']))
    if summary:
        res.summary = torch.from_numpy(_summary(grid, g, r0, r1))
    return res


def _summary(grid, g, r0, r1):
    """engine.SUMMARY_FIELDS of the rays [r0, r1) (sums in ray order: the tests compare the
    floating-point columns with a tolerance)"""
    summ = np.zeros((grid.n_tiles, _abi.RT_SUMMARY_DOUBLES), dtype=np.longdouble)   # order-insensitive sums
    summ[:, [10, 12]], summ[:, [11, 13]] = np.inf, -np.inf
    tile = (np.arange(r0, r1)//grid.rays_per_tile)
    st = g['status']
    for s in range(4):
        np.add.at(summ[:, s + (0 if s == 0 else 0)], tile, st == s)
    np.add.at(summ[:, 4], tile, st > 3)
    ok = st == 0
    x, y = g['abr'][0, ok], g['abr'][1, ok]
    for col, v in ((5, x), (6, y), (7, x*x), (8, y*y), (9, x*y), (14, g['op'][ok])):
        np.add.at(summ[:, col], tile[ok], v)
    np.minimum.at(summ[:, 10], tile[ok], x)
    np.maximum.at(summ[:, 11], tile[ok], x)
    np.minimum.at(summ[:, 12], tile[ok], y)
    np.maximum.at(summ[:, 13], tile[ok], y)
    return summ.astype(np.float64)


def trace_grid_to_host(table, grid, h_abr, chunk_begin=0, chunk_end=None, pieces=8, summary=True,
                       workspace=None, **kwargs):
    chunk_end = grid.n_chunks if chunk_end is None else chunk_end
    n = grid.rays_in_chunks(chunk_begin, chunk_end)
    if not (h_abr.dtype == torch.float64 and h_abr.shape[0] == 2 and h_abr.shape[1] >= n):
        raise ValueError('h_abr must be a pinned float64 tensor [2, >= n] with contiguous rows')
    r = trace_grid(table, grid, chunk_begin, chunk_end, outputs=('abr',), summary=summary,
                   nan_status=True, **kwargs)
    h_abr[:, :n].copy_(r.abr)
    return r.summary, (workspace or {'device': torch.device('cpu')})


def calc_psf(wavefront, ndim, maxdim, device=0):
    from numpy.fft import fftshift, fft2
    W = np.zeros([maxdim, maxdim])
    m2, nd2 = maxdim//2, ndim//2
    W[m2 - (nd2 - 1):m2 + (nd2 + 1), m2 - (nd2 - 1):m2 + (nd2 + 1)] = np.nan_to_num(wavefront)
    phase = np.exp(1j*2*np.pi*W)
    phase[phase == 1] = 0
    AP = abs(fftshift(fft2(fftshift(phase))))**2
    return AP/np.nanmax(AP)


class _NoStream:
    def __init__(self, *a, **k):
        pass

    def wait_stream(self, *a):
        pass

    def synchronize(self):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def _on_cpu(fn):
    def wrapper(*args, **kwargs):
        dev = kwargs.get('device')
        if dev is not None and 'cuda' in str(dev):
            kwargs['device'] = 'cpu'
        return fn(*args, **kwargs)
    return wrapper


def install():
    T.SurfaceTable.from_model = classmethod(_from_model)
    T.SurfaceTable.from_path = classmethod(_from_path)
    E.PupilGrid = DryGrid
    E.trace_bundle, E.trace_grid, E.trace_grid_to_host = trace_bundle, trace_grid, trace_grid_to_host
    A.calc_psf = calc_psf
    # tests (and analyses.spot_diagram) name the CUDA device / pinned memory / streams explicitly
    torch.cuda.synchronize = lambda *a, **k: None
    torch.cuda.current_stream = lambda *a, **k: _NoStream()
    torch.cuda.Stream = _NoStream
    torch.cuda.stream = lambda s: _NoStream()
    torch.cuda.device = _NoStream
    for name in ('empty', 'full', 'zeros', 'ones', 'tensor', 'as_tensor'):
        setattr(torch, name, _on_cpu(getattr(torch, name)))
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    torch.Tensor.is_pinned = lambda self, *a, **k: True
