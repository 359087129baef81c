"""Load the reference's compiled CPython extension modules from oracle/_ref by path
(importing the `stardist` package itself needs csbdeep/skimage/TF).  TEST INFRASTRUCTURE ONLY.

oracle/_ref can only be built where the reference's sources are.  Everywhere else the two modules are
replayed from tests/golden/refcalls/*.npz.xz (an .npz inside an xz stream): the reference's answers to every call the test suite, smoke()
and the fixture scripts make, keyed by a digest of the call's arguments.  A call whose arguments were
never recorded raises KeyError, so a comparison is never skipped silently.  To re-record, build
oracle/_ref and run with STARDIST_ORACLE_RECORD=<dir>; tests/golden/make_refcalls.py merges the files.
"""
import glob, hashlib, importlib.util, io, itertools, lzma, os, ctypes
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_REF = os.path.join(_HERE, "_ref")
REPLAY_DIR = os.path.join(os.path.dirname(_HERE), "tests", "golden", "refcalls")


def _load(name):
    path = os.path.join(_REF, name + ".so")
    if not os.path.exists(path):
        raise FileNotFoundError("%s missing: run `make -C oracle ref` where the reference's sources are" % path)
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _feed(h, a):
    if isinstance(a, np.ndarray) or isinstance(a, np.generic):
        a = np.ascontiguousarray(a)
        h.update(("A%s%s" % (a.dtype.str, a.shape)).encode()); h.update(a.tobytes())
    elif isinstance(a, (tuple, list)):
        h.update(b"(")
        for x in a: _feed(h, x)
        h.update(b")")
    elif isinstance(a, (bool, int, float, str, type(None))):
        h.update(("%s:%r;" % (type(a).__name__, a)).encode())
    else:
        raise TypeError("cannot digest an argument of type %s" % type(a).__name__)


def call_key(module, fn, args, kwargs=None):
    """digest of (module, function, arguments): arrays by dtype, shape and bytes, scalars by type and value"""
    h = hashlib.sha1(("%s.%s" % (module, fn)).encode())
    _feed(h, list(args)); _feed(h, sorted((kwargs or {}).items()))
    return h.hexdigest()[:24]


def _pack(key, out):
    if isinstance(out, tuple):
        return {"%s/t%d" % (key, i): np.asarray(o) for i, o in enumerate(out)}
    return {key: np.asarray(out)}


class _Recorder:
    """wraps a real module: every call's result is also written to $STARDIST_ORACLE_RECORD/<module>_<key>.npz"""
    def __init__(self, name, mod, outdir):
        self._name, self._mod, self._dir = name, mod, outdir
        os.makedirs(outdir, exist_ok=True)

    def __getattr__(self, fn):
        f = getattr(self._mod, fn)
        def call(*args, **kwargs):
            out = f(*args, **kwargs)
            key = call_key(self._name, fn, args, kwargs)
            np.savez_compressed(os.path.join(self._dir, "%s_%s.npz" % (self._name, key)), **_pack(key, out))
            return out
        return call


class _Replay:
    """stands in for a module of oracle/_ref with the recorded answers of tests/golden/refcalls"""
    def __init__(self, name):
        self._name = name
        self._files = [np.load(io.BytesIO(lzma.decompress(open(p, "rb").read()))) for p in replay_files()]

    def _get(self, k):
        for z in self._files:
            if k in z.files: return z[k]
        return None

    def __getattr__(self, fn):
        def call(*args, **kwargs):
            key = call_key(self._name, fn, args, kwargs)
            out = self._get(key)
            if out is not None:
                return out
            parts = list(itertools.takewhile(lambda a: a is not None, (self._get("%s/t%d" % (key, i)) for i in itertools.count())))
            if parts:
                return tuple(parts)
            raise KeyError("%s.%s: no recorded reference result for these arguments (oracle/_ref is not built here; "
                           "see oracle/ref_ext.py)" % (self._name, fn))
        return call


_cache = {}

def _module(name):
    if name not in _cache:
        if os.path.exists(os.path.join(_REF, name + ".so")):
            m = _load(name)
            if os.environ.get("STARDIST_ORACLE_RECORD"):
                m = _Recorder(name, m, os.environ["STARDIST_ORACLE_RECORD"])
        else:
            m = _Replay(name)
        _cache[name] = m
    return _cache[name]

def stardist2d():
    return _module("stardist2d")

def stardist3d():
    return _module("stardist3d")

def sdref():
    if "shim" not in _cache: _cache["shim"] = ctypes.CDLL(os.path.join(_REF, "libsdref.so"))
    return _cache["shim"]

def built():
    """True where oracle/_ref holds the compiled reference modules"""
    return all(os.path.exists(os.path.join(_REF, f)) for f in ("stardist2d.so", "stardist3d.so"))

def replay_files():
    return sorted(glob.glob(os.path.join(REPLAY_DIR, "*.npz.xz")))

def available():
    """True where the reference modules can answer: compiled in oracle/_ref, or replayed from tests/golden/refcalls"""
    return built() or bool(replay_files())
