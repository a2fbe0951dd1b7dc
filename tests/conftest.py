import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="session")
def oracle():
    """The plain-C CPU oracle (oracle/alva_oracle.c), built on demand.  Test infrastructure only."""
    so = os.path.join(ROOT, "oracle", "_build", "libalva_oracle.so")
    srcs = [os.path.join(ROOT, "oracle", f) for f in ("alva_oracle.c", "ba_oracle.c", "klt_oracle.c", "pose_oracle.c", "detect_oracle.c", "match_oracle.c", "init_oracle.c")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    L = C.CDLL(so)
    L.orc_fast_atan2.restype = C.c_float
    L.orc_fast_atan2.argtypes = [C.c_float, C.c_float]
    return L


@pytest.fixture(scope="session")
def ref():
    """The reference itself (oracle/_ref/libalva_ref.so), if it was built in this tree; else None."""
    so = os.path.join(ROOT, "oracle", "_ref", "libalva_ref.so")
    if not os.path.exists(so):
        return None
    L = C.CDLL(so)
    L.ref_config(0, 1)
    return L


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def digest(a):
    """sha256 of an array's dtype, shape and bytes, as uint8[32]: equal digests <=> bit-identical arrays.  A large result that is
    compared bit for bit is recorded in this form."""
    a = np.ascontiguousarray(a)
    return np.frombuffer(hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest(), np.uint8)


RECORD_REFERENCE = os.environ.get("ALVA_RECORD_REFERENCE") == "1"
SAMPLE = 500


class ReferenceResults:
    """What the reference library returned in the tests of one module, so that every comparison with it also runs where it is
    not built.  `get(key, fn)`: with oracle/_ref/libalva_ref.so loaded, fn() calls it and its results (a tuple of arrays) are
    returned; without it, the results it returned when tests/golden/reference/<module>.npz was written (by running the tests
    with the library built and ALVA_RECORD_REFERENCE=1).  The float arrays at the tuple positions in `sample` are recorded as a
    fixed, seeded sample of SAMPLE entries; replayed, the entries not recorded are NaN."""

    def __init__(self, lib, module):
        self.lib, self.path = lib, os.path.join(GOLDEN, "reference", module + ".npz")
        self.stored, self.new = None, {}
        if lib is None and os.path.exists(self.path):
            z = np.load(self.path)
            data = z["data"].tobytes()
            self.stored = {k: np.frombuffer(data, dt, int(np.prod(shape)), off).reshape(shape)
                           for k, dt, shape, off in json.loads(z["index"].tobytes())}

    def available(self):
        return self.lib is not None or self.stored is not None

    def get(self, key, fn, sample=()):
        if self.lib is None:
            if f"{key}#n" not in self.stored:
                raise KeyError(f"{self.path} has no result for {key}: re-record it with the reference built")
            out = []
            for i in range(int(self.stored[f"{key}#n"])):
                if f"{key}#{i}@shape" in self.stored:
                    a = np.full(tuple(self.stored[f"{key}#{i}@shape"]), np.nan)
                    a.flat[self.stored[f"{key}#{i}@at"]] = self.stored[f"{key}#{i}"]
                    out.append(a)
                else:
                    out.append(self.stored[f"{key}#{i}"])
            return tuple(out)
        out = tuple(np.asarray(v) for v in fn())
        if RECORD_REFERENCE:
            self.new[f"{key}#n"] = np.int32(len(out))
            for i, v in enumerate(out):
                if i in sample and v.size > SAMPLE:
                    at = np.sort(np.random.default_rng(0).choice(v.size, SAMPLE, replace=False))
                    self.new.update({f"{key}#{i}@shape": np.array(v.shape), f"{key}#{i}@at": at})
                    v = v.flat[at]
                self.new[f"{key}#{i}"] = v
        return out

    def save(self):
        """one compressed blob + a JSON index: per-array file headers would outweigh the many small results"""
        index, data, off = [], [], 0
        for k, v in self.new.items():
            v = np.asarray(v)
            index.append((k, v.dtype.str, v.shape, off))
            data.append(v.tobytes())
            off += v.nbytes
        os.makedirs(os.path.dirname(self.path), exist_ok=True)
        np.savez_compressed(self.path, index=np.frombuffer(json.dumps(index).encode(), np.uint8),
                            data=np.frombuffer(b"".join(data), np.uint8))


@pytest.fixture(scope="session")
def _reference_results(ref):
    by_module = {}
    yield ref, by_module
    for r in by_module.values():
        if r.new:
            r.save()


@pytest.fixture
def ref_results(request, _reference_results):
    """ReferenceResults of the requesting test's module; skips only when the reference is neither built nor recorded."""
    ref, by_module = _reference_results
    module = request.module.__name__.rsplit(".", 1)[-1]
    if module not in by_module:
        by_module[module] = ReferenceResults(ref, module)
    r = by_module[module]
    if not r.available():
        pytest.skip(f"oracle/_ref/libalva_ref.so not built and {os.path.relpath(r.path, ROOT)} not recorded")
    return r


@pytest.fixture(scope="session")
def gpu_ctx():
    import torch
    if not torch.cuda.is_available():   # a plain `pytest tests` on a machine without a GPU: skip, do not error
        pytest.skip("gpu tests need a CUDA device")
    import alvaar_b200
    ctx = alvaar_b200.Context(0, torch.cuda.current_stream().cuda_stream)
    yield ctx
    ctx.close()
