"""What the original project's own code returned (oracle/ref.py over oracle/_ref/libref.so, which oracle/ref_build.sh compiles
from the original sources), recorded in tests/golden/ref_parity.npz, so that tests/test_ref_parity_cpu.py holds the oracle against
the original on machines that do not have its sources.

Each test gets a Reference: the same calls as oracle/ref.py, answered in call order with what they returned when the file was
recorded.  Outputs that the tests only compare for equality are kept as SHA-256 digests of their dtype, shape and bytes (that keeps
the file small); compare them with same().  The others (those a test indexes, or feeds to the oracle) are kept whole.  To record
again (the whole module, with the original sources at hand for oracle/ref_build.sh):

    SSLPL_RECORD_REFERENCE=1 python -m pytest tests/test_ref_parity_cpu.py
"""
import hashlib
import json
import os
import numpy as np

from conftest import GOLDEN
from oracle import ref as R

PATH = os.path.join(GOLDEN, "ref_parity.npz")
RECORD = os.environ.get("SSLPL_RECORD_REFERENCE") == "1"
DIGESTED = {"orb_extract.0", "orb_extract.1", "orb_pyramid_level", "octree", "features_in_area",
            "search_by_bow.1", "search_by_bow_kf.1", "search_for_triangulation.1", "search_for_initialization.1", "search_for_initialization.2",
            "line_match.1", "Vocabulary.words.0", "Vocabulary.words.1", "Vocabulary.transform.1", "Vocabulary.transform.2",
            "frame_from_image.keys", "frame_from_image.keysUn", "frame_from_image.desc", "frame_from_image.keylines",
            "frame_from_image.ldesc", "frame_from_image.lineeq"}


class Digest:
    """An array known by its dtype, shape and the SHA-256 of its bytes."""

    def __init__(self, hexdigest, shape):
        self.hexdigest, self.shape = hexdigest, tuple(shape)

    def __len__(self):
        return self.shape[0]


def digest(a):
    if isinstance(a, Digest):
        return a.hexdigest
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(repr((a.dtype.descr, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def same(a, b):
    """Bit-equal arrays (either may be a Digest)."""
    return digest(a) == digest(b)


def _pack(obj, path, arrays):
    """A call's result as a JSON skeleton; its whole arrays are added to `arrays` (short member names: the file stays small)."""
    if isinstance(obj, np.ndarray):
        if path in DIGESTED:
            return {"digest": digest(obj), "shape": list(obj.shape)}
        name = f"a{len(arrays)}"
        arrays[name] = obj
        return {"array": name}
    if isinstance(obj, dict):
        return {"dict": {k: _pack(v, f"{path}.{k}", arrays) for k, v in obj.items()}}
    if isinstance(obj, tuple):
        return {"tuple": [_pack(v, f"{path}.{i}", arrays) for i, v in enumerate(obj)]}
    if isinstance(obj, np.generic):
        obj = obj.item()
    assert isinstance(obj, (int, float)), (path, type(obj))
    return {"value": obj}


def _unpack(sk, npz):
    if "array" in sk:
        return npz[sk["array"]]
    if "digest" in sk:
        return Digest(sk["digest"], sk["shape"])
    if "dict" in sk:
        return {k: _unpack(v, npz) for k, v in sk["dict"].items()}
    if "tuple" in sk:
        return tuple(_unpack(v, npz) for v in sk["tuple"])
    return sk["value"]


class Store:
    """The recorded calls of every test of the module: read from the golden file, or (recording) collected and written by save()."""

    def __init__(self):
        if RECORD:
            R.lib()
            self.calls, self.arrays, self.npz = {}, {}, None
        else:
            self.npz = np.load(PATH)
            self.calls = json.loads(str(self.npz["__manifest__"]))

    def reference(self, test):
        if RECORD:
            self.calls[test] = []
        return Reference(self, test)

    def save(self):
        if RECORD:
            np.savez_compressed(PATH, __manifest__=np.array(json.dumps(self.calls)), **self.arrays)


class Reference:
    """oracle/ref.py for one test: run live and recorded, or replayed."""
    cam, CAM640 = staticmethod(R.cam), R.CAM640           # plain helpers: no call into the original

    def __init__(self, store, test):
        self._store, self._test, self._n = store, test, 0

    def _call(self, name, run):
        i = self._n
        self._n += 1
        calls = self._store.calls[self._test]
        if RECORD:
            out = run()
            calls.append({"fn": name, "result": _pack(out, name, self._store.arrays)})
            return out
        assert i < len(calls) and calls[i]["fn"] == name, \
            f"{self._test}: call {i} ({name}) was not recorded in {PATH}; record the module again (see {__name__})"
        return _unpack(calls[i]["result"], self._store.npz)

    def __getattr__(self, name):
        fn = getattr(R, name)
        return lambda *a, **k: self._call(name, lambda: fn(*a, **k))

    def Vocabulary(self, path):
        return _Vocabulary(self, path)


class _Vocabulary:
    def __init__(self, ref, path):
        self._ref, self._v = ref, (R.Vocabulary(path) if RECORD else None)

    def __len__(self):
        return self._ref._call("Vocabulary.__len__", lambda: len(self._v))

    def transform(self, desc, levelsup=4):
        return self._ref._call("Vocabulary.transform", lambda: self._v.transform(desc, levelsup))

    def words(self, desc):
        return self._ref._call("Vocabulary.words", lambda: self._v.words(desc))
