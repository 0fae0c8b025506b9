import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import orc
    return orc.Oracle()


# ---------------------------------------------------------------- T1's answers, stored
# Every call a test makes to the reference's own code (T1 = oracle/_ref, built from the reference's
# sources by oracle/Makefile) goes through T1Answers: where oracle/_ref is built, T1 is called and its
# answer must equal the stored one; elsewhere the stored answer (tests/golden/ref_t1_<module>.xz) is
# returned, after a digest of the call's inputs is checked.  tests/golden/make_golden_t1.py records them.
RECORD_T1 = os.environ.get("MV_RECORD_T1") == "1"


def _digest(name, args):
    import zlib
    h = zlib.crc32(name.encode())
    for a in args:
        if isinstance(a, np.ndarray):
            h = zlib.crc32(np.ascontiguousarray(a).tobytes(), zlib.crc32((a.dtype.str + str(a.shape)).encode(), h))
        elif hasattr(a, "_fields_"):
            h = zlib.crc32(bytes(a), h)
        else:
            h = zlib.crc32(repr(a).encode(), h)
    return h


def _enc(v, blob):
    if isinstance(v, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(v)
        blob += a.tobytes()
        return {"a": [a.dtype.str, list(a.shape), len(blob) - a.nbytes]}
    if isinstance(v, bytes):
        blob += v
        return {"b": [len(blob) - len(v), len(v)]}
    if isinstance(v, tuple):
        return {"t": [_enc(x, blob) for x in v]}
    if isinstance(v, list):
        return [_enc(x, blob) for x in v]
    if isinstance(v, dict):
        return {"d": {k: _enc(x, blob) for k, x in v.items()}}
    assert v is None or isinstance(v, (bool, int, float, str)), type(v)
    return v


def _dec(e, blob):
    if isinstance(e, list):
        return [_dec(x, blob) for x in e]
    if not isinstance(e, dict):
        return e
    if "a" in e:
        dt, shape, off = e["a"]
        return np.frombuffer(blob, dt, int(np.prod(shape)), off).reshape(shape).copy()
    if "b" in e:
        return bytes(blob[e["b"][0]:e["b"][0] + e["b"][1]])
    if "t" in e:
        return tuple(_dec(x, blob) for x in e["t"])
    return {k: _dec(x, blob) for k, x in e["d"].items()}


class T1Answers:
    """T1's answers to the calls one test makes, in call order."""

    def __init__(self, stored):
        self.stored, self.new, self.i = stored, [], 0

    def next(self, name, args, compute=None):
        """`compute` runs T1 (None where T1 is not built) and returns its answer: ndarrays, bytes, numbers,
        and tuples / lists / dicts of them."""
        d = _digest(name, args)
        if RECORD_T1:
            v = compute()
            blob = bytearray()
            self.new.append((d, _enc(v, blob), bytes(blob)))
            return v
        if self.i >= len(self.stored):
            if compute is None:
                pytest.skip("no stored answer of the reference for this call (tests/golden/make_golden_t1.py)")
            return compute()
        sd, enc, blob = self.stored[self.i]
        self.i += 1
        assert sd == d, "the inputs of call %d (%s) are not the ones the stored answer was recorded for" % (self.i, name)
        if compute is None:
            return _dec(enc, blob)
        v = compute()
        b2 = bytearray()
        assert (_enc(v, b2), bytes(b2)) == (enc, blob), "T1's answer differs from the stored one (%s)" % name
        return v


class _T1Store:
    def __init__(self):
        self.modules, self.recorded = {}, {}

    def for_test(self, module, test):
        if module not in self.modules:
            import json
            import lzma
            p = os.path.join(GOLDEN, "ref_t1_%s.xz" % module)
            self.modules[module] = {}
            if os.path.exists(p) and not RECORD_T1:
                with open(p, "rb") as f:
                    meta, blob = lzma.decompress(f.read()).split(b"\0", 1)
                meta = json.loads(meta)
                for t, calls in meta.items():
                    self.modules[module][t] = [(d, e, blob[o:o + n]) for d, e, o, n in calls]
        ans = T1Answers(self.modules[module].get(test, []))
        if RECORD_T1:
            self.recorded.setdefault(module, {})[test] = ans
        return ans

    def save(self):
        """ref_t1_<module>.xz: the JSON index of every test's calls, a NUL, the arrays' bytes; LZMA."""
        import json
        import lzma
        for module, tests in self.recorded.items():
            meta, blob = {}, bytearray()
            for t, ans in sorted(tests.items()):
                meta[t] = []
                for d, e, b in ans.new:
                    meta[t].append([d, e, len(blob), len(b)])
                    blob += b
            with open(os.path.join(GOLDEN, "ref_t1_%s.xz" % module), "wb") as f:
                f.write(lzma.compress(json.dumps(meta).encode() + b"\0" + bytes(blob), preset=9 | lzma.PRESET_EXTREME))


@pytest.fixture(scope="session")
def _t1_store():
    s = _T1Store()
    yield s
    if RECORD_T1:
        s.save()


@pytest.fixture
def t1(request, _t1_store):
    return _t1_store.for_test(request.node.module.__name__, request.node.name)


class T1Calls:
    """Calls of a T1 object (orc.Reference / orc.ReferenceBow or its .lib) answered through T1Answers."""

    def __init__(self, src, answers):
        self._src, self._ans = src, answers

    def __getattr__(self, name):
        if name == "lib":
            return T1Calls(None if self._src is None else self._src.lib, self._ans)
        f = None if self._src is None else getattr(self._src, name)
        return lambda *args: self._ans.next(name, args, None if f is None else (lambda: f(*args)))


@pytest.fixture(scope="session")
def t1_live():
    """The reference's own code (T1) where oracle/_ref is built; when recording without it, the
    restatement that was held bit-equal to it on these inputs (tests/golden/make_golden_t1.py)."""
    from oracle import orc
    orc.build()
    if orc.have_ref():
        return orc.Reference()
    if RECORD_T1:
        from golden.make_golden_t1 import StandInReference
        return StandInReference()
    return None


@pytest.fixture(scope="session")
def t1_lib(t1_live):
    """T1's ctypes library where built; when recording without it, the product library, whose legacy host
    symbols were held bit-equal to T1's on these inputs; else None (the stored answers are used)."""
    from oracle import orc
    if isinstance(t1_live, orc.Reference):
        return t1_live.lib
    if RECORD_T1:
        from golden.make_golden_t1 import product_host_library
        return product_host_library()
    return None


@pytest.fixture
def reference(t1_live, t1):
    """T1: called where built, else its stored answers."""
    return T1Calls(t1_live, t1)


@pytest.fixture(scope="session")
def image0():
    return dict(np.load(os.path.join(GOLDEN, "ref_image0.npz")))


@pytest.fixture(scope="session")
def kat():
    return dict(np.load(os.path.join(GOLDEN, "ref_kat.npz")))


@pytest.fixture(scope="session")
def synth():
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import synth as s
    return s


@pytest.fixture(scope="session")
def tracker():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    return tracking.Tracker(0)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)
