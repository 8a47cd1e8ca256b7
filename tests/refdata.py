"""What the reference computed, stored for the tests that compare against it.

A test that checks this package against the original ray-optics code asks for every value
the reference computes through the ``ref`` fixture: ``want = ref(lambda: <reference call>)``.
Normally ``ref`` reads the values back from tests/golden/reference/<test module>.json.gz, in
the order the test asks for them, so the comparison runs without the reference installed.
Set-up that only those calls need (importing the reference, building its model) goes under
``if ref.live:``.
With ``B200RT_RECORD_REF=1`` and the reference source tree present (oracle/ref_harness.py,
``B200RT_REF_SRC``) it evaluates the calls instead and rewrites the test's entry:

    B200RT_RECORD_REF=1 B200RT_REF_SRC=<ray-optics>/src python -m pytest tests -m "not gpu"

Values are stored exactly: floats as their shortest round-trip text, arrays as their raw
bytes.  Both modes hand the test the stored form (tuples, lists, dicts, numpy arrays and
scalars), so a test sees the same types whether it records or replays.  Values too large
to keep whole (full ray packages) are stored as ``digest()`` and compared as such.

``lens_files()`` is the directory of lens files that ship with ray-optics (its
``src/rayoptics`` layout: codev/tests/*.seq, zemax/tests/*.zmx, models/*.roa ...),
unpacked from tests/golden/reference/lens_files.tar.xz.  ray-optics is Copyright (c)
2017-2025 Michael J. Hayford, BSD 3-Clause License.
"""
import atexit
import base64
import gzip
import hashlib
import json
import os
import shutil
import struct
import tarfile
import tempfile

import numpy as np
import pytest

STORE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference')
RECORD = os.environ.get('B200RT_RECORD_REF') == '1'

_files = {}
_lens_dir = None


def lens_files():
    """Directory holding the lens files of ray-optics (unpacked once per process)."""
    global _lens_dir
    if _lens_dir is None:
        d = tempfile.mkdtemp(prefix='rayoptics_lens_files_')
        atexit.register(shutil.rmtree, d, True)
        with tarfile.open(os.path.join(STORE, 'lens_files.tar.xz')) as t:
            t.extractall(d, filter='data')
        _lens_dir = d
    return _lens_dir


def encode(v):
    if v is None or isinstance(v, (bool, str)):
        return v
    if isinstance(v, (np.bool_,)):
        return bool(v)
    if isinstance(v, bytes):
        return {'__bytes__': base64.b64encode(v).decode('ascii')}
    if isinstance(v, (int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return float(v)
    if isinstance(v, np.ndarray):
        if v.dtype == object:
            return {'__ndobj__': [encode(x) for x in v.ravel()], 'shape': list(v.shape)}
        a = np.ascontiguousarray(v)
        return {'__nd__': base64.b64encode(a.tobytes()).decode('ascii'), 'dtype': a.dtype.str,
                'shape': list(a.shape)}
    if isinstance(v, tuple):
        return {'__tuple__': [encode(x) for x in v]}
    if isinstance(v, list):
        return [encode(x) for x in v]
    if isinstance(v, dict):
        return {'__dict__': [[encode(k), encode(x)] for k, x in v.items()]}
    raise TypeError(f'cannot store a {type(v).__name__} as a reference value: reduce it to plain data')


def decode(v):
    if isinstance(v, list):
        return [decode(x) for x in v]
    if not isinstance(v, dict):
        return v
    if '__bytes__' in v:
        return base64.b64decode(v['__bytes__'])
    if '__nd__' in v:
        a = np.frombuffer(base64.b64decode(v['__nd__']), dtype=np.dtype(v['dtype']))
        return a.reshape(v['shape']).copy()
    if '__ndobj__' in v:
        a = np.empty(len(v['__ndobj__']), dtype=object)
        a[:] = [decode(x) for x in v['__ndobj__']]
        return a.reshape(v['shape'])
    if '__tuple__' in v:
        return tuple(decode(x) for x in v['__tuple__'])
    return {_key(decode(k)): decode(x) for k, x in v['__dict__']}


def _canon(v, out):
    if isinstance(v, np.ndarray) and v.dtype != object:
        v = v.tolist()
    if v is None:
        out.append(b'N')
    elif isinstance(v, str):
        out.append(b'S' + v.encode() + b'\0')
    elif isinstance(v, (list, tuple, np.ndarray)):
        out.append(b'[')
        for x in v:
            _canon(x, out)
        out.append(b']')
    else:
        x = float(v)
        out.append(b'F' + (b'nan' if x != x else struct.pack('<d', x + 0.0)))


def digest(v):
    """SHA-256 of a nested value, equal for two values exactly when they hold the same numbers
    (compared with ==, NaN equal to NaN) in the same nesting: lists, tuples and arrays alike."""
    out = []
    _canon(v, out)
    return hashlib.sha256(b''.join(out)).hexdigest()


def _key(k):
    return tuple(_key(x) for x in k) if isinstance(k, (list, tuple)) else k


def _path(module):
    return os.path.join(STORE, module + '.json.gz')


def _load(module):
    if module not in _files:
        try:
            with gzip.open(_path(module), 'rt') as f:
                _files[module] = json.load(f)
        except FileNotFoundError:
            _files[module] = {}
    return _files[module]


def _save(module):
    os.makedirs(STORE, exist_ok=True)
    text = json.dumps(_files[module], sort_keys=True, separators=(',', ':'))
    with open(_path(module), 'wb') as raw, gzip.GzipFile(fileobj=raw, mode='wb', mtime=0) as f:
        f.write(text.encode())


class Recording:
    def __init__(self, module, test):
        self.module, self.test = module, test
        self.live = RECORD          # set-up that only the reference calls need runs only when True
        if RECORD:
            from oracle import ref_harness as rh
            if not rh.available():
                raise RuntimeError(f'B200RT_RECORD_REF=1 needs the reference source tree at {rh.REF_SRC}')
            self.values = []
        else:
            stored = _load(module)
            if test not in stored:
                pytest.fail(f'no stored reference values for {module}::{test} in {_path(module)} '
                            '(record them with B200RT_RECORD_REF=1)')
            self.values = stored[test]
        self.pos = 0

    def __call__(self, compute):
        """The reference's value: ``compute()`` when recording, the stored value otherwise."""
        if RECORD:
            self.values.append(encode(compute()))
        elif self.pos >= len(self.values):
            pytest.fail(f'{self.module}::{self.test} asks for more reference values than were recorded')
        v = decode(self.values[self.pos])
        self.pos += 1
        return v

    def digest(self, compute):
        """``digest()`` of the reference's value, for values too large to store whole"""
        return self(lambda: digest(compute()))

    def finish(self):
        if RECORD:
            _load(self.module)[self.test] = self.values
            _save(self.module)


@pytest.fixture
def ref(request):
    rec = Recording(request.node.module.__name__, request.node.name)
    yield rec
    rec.finish()
