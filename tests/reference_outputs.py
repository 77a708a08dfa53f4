"""What the original PL-SVO code (oracle/_ref: its own translation units) computes on the seeded inputs the tests build.

oracle/_ref can only be built where the original sources are.  Everywhere else the tests compare with the record of an
earlier run, tests/golden/reference_outputs.npz.  Outputs compared bit for bit are stored as 128-bit SHA-256 digests
(NaN == NaN and -0.0 == 0.0, as numpy.testing.assert_array_equal has it), which keeps the record small; the small
integer outputs a test reads (a status, a flag) are stored whole.  Every record carries a digest of its inputs, so inputs that a generator
no longer reproduces fail as such instead of as a parity failure.

Where oracle/_ref is built, the live outputs are used and checked against the record.  PLSVO_RECORD_REFERENCE=1 rewrites
the record from the live run instead:  PLSVO_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"
"""
import ctypes
import hashlib
import os

import numpy as np

import oracle_lib

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")
RECORD = bool(os.environ.get("PLSVO_RECORD_REFERENCE"))
_store = None


def _load():
    """{name: digest (hex str) or whole array}"""
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(PATH):
            z = np.load(PATH)
            _store = {str(n): d.tobytes().hex() for n, d in zip(z["digest_names"], z["digests"])}
            _store.update({k[len("array|"):]: z[k] for k in z.files if k.startswith("array|")})
    return _store


def _put(name, value):
    store = _load()
    store[name] = value
    names = sorted(k for k, v in store.items() if isinstance(v, str))
    digests = np.array([np.frombuffer(bytes.fromhex(store[k]), np.uint8) for k in names]).reshape(len(names), 16)
    arrays = {"array|" + k: v for k, v in sorted(store.items()) if not isinstance(v, str)}
    np.savez_compressed(PATH, digest_names=np.array(names), digests=digests, **arrays)


def _feed(h, x):
    if isinstance(x, np.ndarray):
        h.update(f"{x.dtype.str}{x.shape}".encode())
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, dict):
        for k in sorted(x, key=repr):
            _feed(h, k)
            _feed(h, x[k])
    elif isinstance(x, (list, tuple)):
        for v in x:
            _feed(h, v)
    elif isinstance(x, ctypes.Structure):
        h.update(bytes(x))
    elif hasattr(x, "detach"):  # torch tensor
        _feed(h, x.detach().cpu().numpy())
    elif hasattr(x, "__dict__") and not isinstance(x, type):  # dataclass batches, cameras
        _feed(h, vars(x))
    else:
        h.update(repr(x).encode())


def digest(x) -> str:
    if isinstance(x, np.ndarray) and x.dtype.kind in "fc":
        x = np.where(np.isnan(x), np.nan, x + 0.0).astype(x.dtype)  # one NaN, and -0.0 -> 0.0
    h = hashlib.sha256()
    _feed(h, x)
    return h.hexdigest()[:32]


class Reference:
    """Reference(key, inputs, run[, names]): run() runs the original code on `inputs` (any nesting of arrays, batches and
    parameters) and returns {name: array}, or an object whose attributes `names` are the outputs; `key` names the record."""

    def __init__(self, key, inputs, run, names=None):
        self.key = key
        self.live = None
        if oracle_lib.ref_available():
            out = run()
            self.live = {k: np.asarray(out[k] if names is None else getattr(out, k)) for k in (names or out)}
        assert self.live is not None or not RECORD, "PLSVO_RECORD_REFERENCE=1 needs oracle/_ref"
        d = digest(inputs)
        if RECORD:
            _put(f"{key}|inputs", d)
        else:
            stored = _load().get(f"{key}|inputs")
            assert stored is not None, f"{key}: no recorded reference outputs in {PATH}"
            assert str(stored) == d, f"{key}: the inputs differ from those the recorded reference outputs were computed from"

    def array(self, name):
        """The whole output `name` (for small integer outputs a test reads)."""
        rec = f"{self.key}|{name}"
        if RECORD:
            _put(rec, self.live[name])
        elif self.live is not None:
            np.testing.assert_array_equal(self.live[name], _load()[rec], err_msg=f"{rec}: live run != record")
        return self.live[name] if self.live is not None else _load()[rec]

    def assert_equal(self, name, got, select=None, err_msg=""):
        """got == the output `name` (restricted to `select`, e.g. a mask) bit for bit."""
        tag = name if select is None else f"{name}[{digest(np.asarray(select))[:12]}]"
        rec = f"{self.key}|{tag}#sha256"
        if self.live is not None:
            want = self.live[name] if select is None else self.live[name][select]
            np.testing.assert_array_equal(got, want, err_msg=err_msg or name)
            if RECORD:
                _put(rec, digest(want))
                return
        stored = _load().get(rec)
        assert stored is not None, f"{rec}: not in the record {PATH}"
        assert digest(np.asarray(got)) == str(stored), f"{self.key}: {err_msg or name} differs from the original code's output"
