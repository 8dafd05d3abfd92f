"""Recorded outputs of the reference that tests compare this project with.

A test that checks the engine against the reference (the unmodified x42 meters.lv2 sources, compiled into oracle/_ref by
oracle/Makefile where those sources are at hand) drives the reference side through a tape:

    def test_x(reftape):                             # tests/conftest.py: one tape per test node (parameters included)
        r = reftape.obj(lambda: O.Ebu(4, kind="reference"))
        r.process(blk)                               # a no-op when the reference is replayed
        assert np.array_equal(ours, reftape.ref(lambda: r.read()))

With oracle/_ref present the reference runs live.  Without it, every value the test compares with is replayed, in order, from
tests/golden/ref/<test module>.npz, so the comparison itself stays in the suite.  Values are stored as they are; bulk byte
strings pass through `t.digest()` and are compared by their BLAKE2b-128 digest.

B200M_REF_TAPE=replay forces the replay although oracle/_ref exists; B200M_REF_TAPE=<directory> runs the reference live and
writes the tapes into <directory>/<test module>.npz (copy them to tests/golden/ref/ to update the recording).
"""
import hashlib
import json
import os

import numpy as np

import _oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")


class _Absent:
    """stands in for a reference object while its outputs are replayed: every attribute, call and index is a no-op"""

    def __getattr__(self, name):
        return self

    def __call__(self, *a, **k):
        return self

    def __getitem__(self, k):
        return self


def digest(b):
    return hashlib.blake2b(bytes(b), digest_size=16).hexdigest()


class Tape:
    def __init__(self, module, name):
        self.module, self.name = module, name
        mode = os.environ.get("B200M_REF_TAPE", "")
        self.record_dir = mode if mode not in ("", "replay") else None
        self.live = mode != "replay" and O.available("reference")
        if self.record_dir and not self.live:
            raise RuntimeError("recording needs oracle/_ref (make -C oracle ref)")
        self.values, self.pos = [], 0
        if not self.live:
            path = os.path.join(GOLD, module + ".npz")
            with np.load(path) as z:
                if name + "/meta" not in z.files:
                    raise KeyError("%s has no recording of %s" % (path, name))
                meta, blob = json.loads(bytes(z[name + "/meta"]).decode()), z[name + "/blob"].tobytes()
            off = 0
            for dt, shape in meta:
                a = np.frombuffer(blob, np.dtype(dt), int(np.prod(shape, dtype=np.int64)), off).reshape(shape)
                off += a.nbytes
                self.values.append(a.copy())

    def obj(self, make, n=None):
        """the reference object `make()` builds, or stand-ins for it (n of them for a tuple) when replaying"""
        if self.live:
            return make()
        return _Absent() if n is None else tuple(_Absent() for _ in range(n))

    def ref(self, get):
        """the reference's value get() (converted to an array), live or replayed"""
        if self.live:
            v = np.array(get())
            self.values.append(v)
            return v
        if self.pos >= len(self.values):
            raise IndexError("the recording of %s::%s ends after %d values" % (self.module, self.name, self.pos))
        v = self.values[self.pos]
        self.pos += 1
        return v

    def refs(self, get, n):
        """the n values of the tuple get() returns, live or replayed"""
        if self.live:
            return [self.ref(lambda: v) for v in get()]
        return [self.ref(None) for _ in range(n)]

    def digest(self, get):
        """digest() of the reference's byte string get(), live or replayed"""
        return bytes(self.ref(lambda: np.frombuffer(digest(get()).encode(), np.uint8))).decode()

    def close(self):
        """after the test passed: a replay must have used the whole recording; a recording run writes it"""
        if not self.live:
            assert self.pos == len(self.values), "%s::%s compared %d of %d recorded values" % (self.module, self.name, self.pos, len(self.values))
            return
        if not self.record_dir:
            return
        os.makedirs(self.record_dir, exist_ok=True)
        path = os.path.join(self.record_dir, self.module + ".npz")
        old = {}
        if os.path.exists(path):
            with np.load(path) as z:
                old = {k: z[k] for k in z.files}
        vals = [np.array(v, order="C") for v in self.values]
        meta = json.dumps([[v.dtype.str, list(v.shape)] for v in vals]).encode()
        old[self.name + "/meta"] = np.frombuffer(meta, np.uint8)
        old[self.name + "/blob"] = np.frombuffer(b"".join(v.tobytes() for v in vals), np.uint8)
        np.savez_compressed(path, **old)
