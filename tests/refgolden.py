"""Stored answers of the reference's own code for the tests that pin the oracle against it.

The libraries under oracle/_ref/ are compiled from the reference tree (oracle/Makefile), which a checkout of this repository does not have.  The
tests therefore call them through `load(LIB, __name__)`:

  SGS_RECORD_REF=1 python -m pytest tests/test_*_ref.py   # with the libraries built: every call runs the real code and its results are stored
  python -m pytest tests/test_*_ref.py                    # the stored results are replayed; no reference tree and no library needed

A call is identified by the function's name, a digest of its inputs (array contents, scalars, file names) and its occurrence among calls with the
same identity.  What is stored is what the call produced: its return value, every array and by-reference scalar it changed and every file it wrote.
A call whose inputs were never recorded fails: the stored answers are stale for the code that asks, and must be recorded again.  Arrays are passed
as `ptr(a)` (a c_void_p that keeps its array) so that the recorder knows what a call wrote."""
import atexit
import ctypes as C
import glob
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref')
RECORD = os.environ.get('SGS_RECORD_REF') == '1'
SHARD_BYTES = 900 * 1024            # raw bytes of arrays per stored file: every file stays below 1 MB


class Ptr(C.c_void_p):
    """Pointer to an array's data that keeps the array."""


def ptr(a):
    assert a.flags['C_CONTIGUOUS']
    p = Ptr(a.ctypes.data)
    p.array = a
    return p


def _is_ref(x):
    return type(x).__name__ == 'CArgObject'


def _is_path(x):
    return isinstance(x, bytes) and os.path.isabs(x.decode(errors='replace'))


def _digest(name, args):
    h = hashlib.sha256(name.encode())
    for x in args:
        if isinstance(x, Ptr):
            h.update(b'P%s%d' % (x.array.dtype.str.encode(), x.array.nbytes)); h.update(x.array.tobytes())
        elif _is_ref(x):
            h.update(b'R' + repr(x._obj.value).encode())
        elif isinstance(x, C._SimpleCData):
            h.update(b'S' + repr(x.value).encode())
        elif _is_path(x):
            h.update(b'F' + os.path.basename(x))      # where a temporary file lies is not an input
        else:
            h.update(b'V' + repr(x).encode())
    return h.hexdigest()[:24]


def _written_rows(a, before):
    """The array up to the last row the call changed (rows after it are the caller's, unchanged)."""
    b = np.frombuffer(before, np.uint8).reshape(a.shape[0] if a.ndim else 1, -1)
    now = np.frombuffer(a.tobytes(), np.uint8).reshape(b.shape)
    last = int(np.nonzero((now != b).any(1))[0][-1]) + 1
    return a.reshape(b.shape[0], *a.shape[1:])[:last].copy()


class _Store:
    def __init__(self, module):
        self.module = module
        self.seen = {}
        self.records = []              # record mode: (key, meta, arrays)
        self.index = None              # replay mode: key -> (meta, npz)

    def next_key(self, name, args):
        d = _digest(name, args)
        k = self.seen.get((name, d), 0)
        self.seen[(name, d)] = k + 1
        return '%s:%s:%d' % (name, d, k)

    def lookup(self, key):
        if self.index is None:
            self.index = {}
            for f in sorted(glob.glob(os.path.join(GOLDEN, self.module + '.*.npz'))):
                z = np.load(f)
                for k, m in json.loads(bytes(z['__meta__']).decode()).items():
                    self.index[k] = (m, z)
        if key not in self.index:
            raise AssertionError('%s: no recorded reference result for %s (tests/golden/ref is stale for these inputs: record it again with SGS_RECORD_REF=1 '
                                 'and the reference libraries built)' % (self.module, key))
        return self.index[key]

    def save(self):
        for f in glob.glob(os.path.join(GOLDEN, self.module + '.*.npz')):
            os.remove(f)
        os.makedirs(GOLDEN, exist_ok=True)
        shard, meta, arrays, size = 0, {}, {}, 0
        for key, m, arrs in self.records + [(None, None, None)]:
            if meta and (key is None or size > SHARD_BYTES):
                arrays['__meta__'] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), np.uint8)
                np.savez_compressed(os.path.join(GOLDEN, '%s.%d.npz' % (self.module, shard)), **arrays)
                shard, meta, arrays, size = shard + 1, {}, {}, 0
            if key is None:
                break
            names = {}
            for j, a in arrs.items():
                h = hashlib.sha256(a.dtype.str.encode() + a.tobytes()).hexdigest()[:16]      # identical results are stored once
                names[j] = 'd' + h
                if names[j] not in arrays:
                    arrays[names[j]] = a
                    size += a.nbytes
            meta[key] = dict(m, arrays=names)


class _Function:
    def __init__(self, lib, name):
        self.lib, self.name, self.restype = lib, name, C.c_int

    def __call__(self, *args):
        st = self.lib.store
        key = st.next_key(self.name, args)
        if RECORD:
            before = {j: x.array.tobytes() for j, x in enumerate(args) if isinstance(x, Ptr)}
            refs = {j: x._obj.value for j, x in enumerate(args) if _is_ref(x)}
            files = {j: (open(x, 'rb').read() if os.path.exists(x) else None) for j, x in enumerate(args) if _is_path(x)}
            fn = getattr(self.lib.real, self.name)
            fn.restype = self.restype
            ret = fn(*args)
            arrs = {'a%d' % j: _written_rows(args[j].array, b) for j, b in before.items() if args[j].array.tobytes() != b}
            arrs.update({'f%d' % j: np.frombuffer(open(args[j], 'rb').read(), np.uint8).copy() for j, b in files.items()
                         if os.path.exists(args[j]) and open(args[j], 'rb').read() != b})
            meta = {'ret': ret, 'refs': {str(j): args[j]._obj.value for j, v in refs.items() if args[j]._obj.value != v}}
            st.records.append((key, meta, arrs))
            return ret
        meta, z = st.lookup(key)
        for j, v in meta['refs'].items():
            args[int(j)]._obj.value = v
        for tag, name in meta['arrays'].items():
            j = int(tag[1:])
            if tag[0] == 'a':
                rows = z[name]
                args[j].array[:len(rows)] = rows.reshape((len(rows),) + args[j].array.shape[1:])
            else:
                with open(args[j], 'wb') as f:
                    f.write(z[name].tobytes())
        return meta['ret']


class Library:
    """Stands for one reference library: records its calls or replays them (see the module's docstring)."""

    def __init__(self, path, module):
        self.store = _Store(module)
        self.fns = {}
        self.real = None
        if RECORD:
            if not os.path.exists(path):
                raise RuntimeError('SGS_RECORD_REF=1 needs %s (build() makes it when the reference tree is present)' % path)
            self.real = C.CDLL(path)
            atexit.register(self.store.save)

    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)
        if name not in self.fns:
            self.fns[name] = _Function(self, name)
        return self.fns[name]


_LIBS = {}


def load(path, module):
    """The library at `path` for the test module `module` (its stored answers are tests/golden/ref/<module>.*.npz)."""
    module = module.rsplit('.', 1)[-1]
    if (path, module) not in _LIBS:
        _LIBS[(path, module)] = Library(path, module)
    return _LIBS[(path, module)]
