"""Regression snapshots for the tests whose checker is the reference-compiled library (oracle/_ref/libbshot_ref.so).

That library can only be built where the original project's sources are at hand, and without it those tests used to
skip.  They now compare with two things:
 * the reference's own output, live, wherever oracle/_ref is built (the comparison these tests were written for);
 * everywhere, a snapshot of what this project's implementation under test returned for the same inputs
   (tests/golden/output_snapshots.json).  A snapshot says that the output has not changed since it was recorded; it
   says nothing about agreement with the reference.  The entries of output_snapshots.json were recorded on a B200
   from the device preprocessor and from the CPU oracle where no reference-compiled library was available.

A snapshot is stored as shape, dtype, SHA-256 and first rows (the rows only make a failure readable), under a key
made from the name of the call and a digest of its inputs; the comparison is bit for bit.  Recording runs the
implementation under test and writes what it returns, so record only from a build whose output is known to be right:
    BSHOT_RECORD_SNAPSHOTS=1 python -m pytest tests/test_ref_pin.py tests/test_preprocess.py tests/test_host_shim.py"""
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "output_snapshots.json")
RECORD = bool(os.environ.get("BSHOT_RECORD_SNAPSHOTS"))
HEAD_ROWS = 4


def _key(name, args):
    h = hashlib.sha256()
    for a in args:
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a)
            h.update(f"{a.dtype.str}{a.shape}".encode())
            h.update(a.tobytes())
        else:
            h.update(repr(a).encode())
        h.update(b"|")
    return f"{name}:{h.hexdigest()[:24]}"


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class Snapshot:
    """one stored output"""

    def __init__(self, shape, dtype, sha256, head, source):
        self.shape, self.dtype, self.sha256, self.head, self.source = tuple(shape), dtype, sha256, head, source

    @classmethod
    def of(cls, a, source):
        a = np.ascontiguousarray(a)
        return cls(a.shape, a.dtype.str, _sha(a), a[:HEAD_ROWS].tolist(), source)

    def record(self):
        return dict(shape=list(self.shape), dtype=self.dtype, sha256=self.sha256, head=self.head, source=self.source)

    def __len__(self):
        return self.shape[0]

    def check(self, a, what="output"):
        """bit-for-bit equality of `a` with the stored output"""
        a = np.ascontiguousarray(a)
        assert a.dtype.str == self.dtype, f"{what}: dtype {a.dtype.str}, snapshot {self.dtype}"
        assert a.shape == self.shape, f"{what}: shape {a.shape}, snapshot {self.shape}"
        if _sha(a) == self.sha256:
            return
        head = np.array(self.head, dtype=self.dtype).reshape((-1,) + self.shape[1:])
        rows = [i for i in range(len(head)) if a[i].tobytes() != head[i].tobytes()]
        where = f"first at row {rows[0]}: {a[rows[0]]} vs {head[rows[0]]}" if rows else f"beyond the first {len(head)} rows"
        raise AssertionError(f"{what} differs from the snapshot of the {self.source} ({where})")


class Expected:
    """what a call must return: its snapshot and, where the reference-compiled library is built, the reference's output"""

    def __init__(self, snapshot, reference=None):
        self.snapshot, self.reference = snapshot, reference

    def __len__(self):
        return len(self.snapshot)

    def check(self, a, what="output"):
        if self.reference is not None:
            r = np.ascontiguousarray(self.reference)
            a = np.ascontiguousarray(a)
            assert a.shape == r.shape and a.tobytes() == r.tobytes(), f"{what} differs from the reference's output"
        self.snapshot.check(a, what)


class Snapshots:
    """the snapshots of one test module"""

    def __init__(self, path=PATH):
        self.path = path
        self.entries = json.load(open(path)) if os.path.exists(path) else {}
        self.recorded = {}

    def expect(self, name, args, implementation, source, reference=None):
        """Expected (or a dict of them for a dict result) for `name(*args)`: the stored snapshot -- recorded from
        `implementation(*args)` when recording -- and `reference(*args)` where a reference is given"""
        k = _key(name, args)
        if RECORD:
            out = implementation(*args)
            snap = ({f: Snapshot.of(v, source) for f, v in out.items()} if isinstance(out, dict) else Snapshot.of(out, source))
            self.recorded[k] = {f: s.record() for f, s in snap.items()} if isinstance(snap, dict) else snap.record()
        elif k not in self.entries:
            raise AssertionError(f"{name}: no snapshot for these inputs in {os.path.basename(self.path)} "
                                 "(record one with BSHOT_RECORD_SNAPSHOTS=1, see tests/golden/snapshots.py)")
        else:
            e = self.entries[k]
            snap = Snapshot(**e) if "sha256" in e else {f: Snapshot(**v) for f, v in e.items()}
        ref = None if reference is None else reference(*args)
        if isinstance(snap, dict):
            return {f: Expected(s, None if ref is None else ref[f]) for f, s in snap.items()}
        return Expected(snap, ref)

    def save(self):
        if not self.recorded:
            return
        entries = json.load(open(self.path)) if os.path.exists(self.path) else {}
        entries.update(self.recorded)
        with open(self.path, "w") as f:   # one entry per line
            f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(entries.items())) + "\n}\n")


class ExpectedPreprocessing:
    """expected output of Preprocessor::run: snapshot of the device preprocessor, plus the reference's preprocess.cpp
    (oracle.ref_preprocess) where oracle/_ref is built"""

    def __init__(self, snapshots, oracle, device_ctx):
        self.snapshots, self.device = snapshots, device_ctx
        self.reference = oracle.ref_preprocess if oracle.ref_lib() is not None else None

    def preprocess(self, azimuth_deg, vertical_deg, distance, ring_deg, vert_init=-0.6, lowpt_th=-1950.0, select=None,
                   save_selected=True):
        args = (np.ascontiguousarray(azimuth_deg, dtype=np.float64), np.ascontiguousarray(vertical_deg, dtype=np.float64),
                np.ascontiguousarray(distance, dtype=np.uint16), np.ascontiguousarray(ring_deg, dtype=np.float64),
                float(vert_init), float(lowpt_th), None if select is None else np.ascontiguousarray(select, dtype=np.int32),
                bool(save_selected))
        return self.snapshots.expect("preprocess", args, self.device.preprocess, "device preprocessor (bshot_preprocess)",
                                     self.reference)
