"""The original project's answers to the calls the tests make, replayed from golden data.

The compiled reference (oracle/_ref, built by oracle/build_ref.sh) exists only where the original sources lie.  So the
`ref_oracle` fixture answers every call from tests/golden/reference_calls_v1.npz instead: one record per distinct call,
keyed by the oracle.ref function and its arguments.  The comparisons with the reference thus run on every machine.

After adding or changing a call to the reference in a test, record the answers again by running the whole suite, GPU
tests included, where the reference is built:

    DGB200_RECORD_REFERENCE=tests/golden/reference_calls_v1.npz python -m pytest tests

Every call is then answered by the compiled reference, and all answers are written to that file when the session ends.
"""
import hashlib
import inspect
import io
import os

import numpy as np

from oracle import ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls_v1.npz")


def call_key(name, args, kwargs):
    """20-byte key of the call ref.<name>(*args, **kwargs), defaults filled in.  Float arrays enter rounded to float32:
    inputs generated on another CPU may differ in the last bits of a double."""
    bound = inspect.signature(getattr(ref, name)).bind(*args, **kwargs)
    bound.apply_defaults()
    h = hashlib.sha1(name.encode())
    for pname, v in bound.arguments.items():
        h.update(b"|" + pname.encode() + b"=")
        if isinstance(v, (bool, np.bool_, int, np.integer)):
            h.update(b"i%d" % int(v))
        elif isinstance(v, (float, np.floating)):
            h.update(b"f" + repr(float(v)).encode())
        else:
            a = np.ascontiguousarray(v)
            if a.dtype.kind == "f":
                a = a.astype(np.float32)
            h.update(("a%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes())
    return h.digest()


def _pack(out):
    items = out if isinstance(out, tuple) else (out,)
    buf = io.BytesIO()
    for x in items:
        np.save(buf, np.asarray(x), allow_pickle=False)
    return isinstance(out, tuple), len(items), buf.getvalue()


def _unpack(is_tuple, count, blob):
    f = io.BytesIO(blob)
    items = []
    for _ in range(count):
        a = np.load(f, allow_pickle=False)
        items.append(a.item() if a.ndim == 0 else a)
    return tuple(items) if is_tuple else items[0]


class ReferenceCalls:
    """The call surface of oracle.ref.  Answers from the recorded golden data, or, with record_to set, from the
    compiled reference, keeping every answer for save()."""

    def __init__(self, record_to=None):
        self.record_to = record_to
        self.records = {}
        if record_to:
            if not ref.available():
                raise RuntimeError("recording needs the compiled reference (oracle/build_ref.sh)")
            return
        with np.load(GOLDEN) as z:
            keys, is_tuple, counts, offsets, blob = (z[k] for k in ("keys", "is_tuple", "counts", "offsets", "blob"))
        blob = blob.tobytes()
        for i, k in enumerate(keys):
            self.records[k.tobytes()] = (bool(is_tuple[i]), int(counts[i]), blob[offsets[i]:offsets[i + 1]])

    def available_final_lsq(self):
        return ref.available_final_lsq() if self.record_to else True

    def __getattr__(self, name):
        fn = getattr(ref, name)

        def call(*args, **kwargs):
            key = call_key(name, args, kwargs)
            if self.record_to:
                out = fn(*args, **kwargs)
                self.records[key] = _pack(out)
                return out
            if key not in self.records:
                raise LookupError("no recorded answer of the reference to this call of oracle.ref.%s: record the answers "
                                  "again (see tests/reference_calls.py)" % name)
            return _unpack(*self.records[key])
        return call

    def save(self):
        keys = sorted(self.records)
        recs = [self.records[k] for k in keys]
        offsets = np.cumsum([0] + [len(r[2]) for r in recs])
        np.savez_compressed(self.record_to, keys=np.frombuffer(b"".join(keys), dtype=np.uint8).reshape(-1, 20),
                            is_tuple=np.array([r[0] for r in recs], dtype=np.uint8),
                            counts=np.array([r[1] for r in recs], dtype=np.uint8), offsets=offsets.astype(np.int64),
                            blob=np.frombuffer(b"".join(r[2] for r in recs), dtype=np.uint8))
