"""Recorded answers of the reference's own ikd-Tree for the tests that compare with it (test infrastructure only).

The reference's sources are not part of this repository, so a test that checks the device map against the reference's
tree runs against a tape: the calls the test made on that tree, in order, each with a digest of its arguments and what
the tree returned.  A call whose arguments differ from the recorded ones fails the test -- the tape does not describe
that input -- instead of answering with a stale result.

Tapes are tests/golden/tapes/<name>.npz.  To (re)record them, build oracle/_ref (oracle/Makefile, needs the reference's
sources) and run the tests that use them with FAST_LIO_RECORD_TAPES=<directory>; they then call the live tree and write
their tapes there.  Tapes of GPU tests whose arguments come from the device (map_incremental's points) must be recorded
on a GPU.

Point arrays the tree returns (flatten(), the neighbours of knn() and update_iterated()) are copies of points it was
given -- the initial map and every add() batch -- and are stored as row numbers into those.  knn()'s squared distances
are recomputed from its neighbours in the tree's own float32 arithmetic; recording checks that they come out bit for bit.
"""
from __future__ import annotations

import hashlib
import os
import types

import numpy as np

TAPES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tapes")
RECORD_DIR = os.environ.get("FAST_LIO_RECORD_TAPES")


def _digest(args) -> str:
    h = hashlib.sha256()
    for a in args:
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a)
            h.update(f"{a.dtype.str}{a.shape}".encode())
            h.update(a.tobytes())
        else:
            h.update(repr(a).encode())
        h.update(b"|")
    return h.hexdigest()[:32]


def _sq_dist(q4, pts, cnt):
    """float32 (dx^2 + dy^2) + dz^2 per neighbour, the ikd-Tree's calc_dist; inf past the number found."""
    d = pts[..., :3] - q4[:, None, :3]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    d2[np.arange(pts.shape[1])[None, :] >= cnt[:, None]] = np.inf
    return d2


class ReferenceTree:
    """Stands in for oracle.bind.KdTree(pts, "reference", downsample): the same methods, answered from the tape `name`."""

    def __init__(self, name: str, pts4, downsample: float = 0.5):
        pts4 = np.ascontiguousarray(pts4, dtype=np.float32)
        self.name = name
        self.given = [pts4]
        self.n = 0
        if RECORD_DIR:
            from oracle import bind
            assert bind.have_ref(), "recording a tape needs oracle/_ref (the reference's ikd-Tree)"
            self.live = bind.KdTree(pts4, "reference", downsample=downsample)
            self.rec, self.args = {}, []
        else:
            self.live = None
            self.tape = np.load(os.path.join(TAPES, name + ".npz"))
        self._call("create", (pts4, downsample), lambda: {})

    # --- what the tests call
    def add(self, pts4, downsample_on: bool) -> int:
        pts4 = np.ascontiguousarray(pts4, dtype=np.float32)
        out = self._call("add", (pts4, bool(downsample_on)), lambda: {"n": self.live.add(pts4, downsample_on)})
        self.given.append(pts4)
        return int(out["n"])

    def delete_boxes(self, boxes6) -> int:
        boxes6 = np.ascontiguousarray(boxes6, dtype=np.float32).reshape(-1, 6)
        return int(self._call("delete_boxes", (boxes6,), lambda: {"n": self.live.delete_boxes(boxes6)})["n"])

    def validnum(self) -> int:
        return int(self._call("validnum", (), lambda: {"n": self.live.validnum()})["n"])

    def flatten(self) -> np.ndarray:
        """The stored points, in the order they were given (callers compare sorted rows)."""
        return self._call("flatten", (), lambda: {"rows": self.live.flatten()})["rows"]

    def knn(self, q4, k: int = 5):
        q4 = np.ascontiguousarray(q4, dtype=np.float32)

        def run():
            pts, d2, cnt = self.live.knn(q4, k)
            assert np.array_equal(d2, _sq_dist(q4, pts, cnt)), "the tree's distances differ from calc_dist restated"
            return {"points": pts, "cnt": cnt}

        out = self._call("knn", (q4, k), run)
        return out["points"], _sq_dist(q4, out["points"], out["cnt"]), out["cnt"]

    def update_iterated(self, scan4, x26, P, max_iter, R=0.001, limit=0.001, extrinsic_est_en=0):
        """oracle.bind.update_iterated on this tree: x, P, nearest and nearest_cnt of the result."""
        from oracle import bind
        scan4 = np.ascontiguousarray(scan4, dtype=np.float32)
        x26, P = np.asarray(x26, dtype=np.float64), np.asarray(P, dtype=np.float64)

        def run():
            o = bind.update_iterated(self.live, scan4, x26, P, max_iter, R, limit, extrinsic_est_en)
            return {"x": o.x, "P": o.P, "points": o.nearest, "cnt": o.nearest_cnt}

        out = self._call("update_iterated", (scan4, x26, P, max_iter, R, limit, extrinsic_est_en), run)
        return types.SimpleNamespace(x=out["x"], P=out["P"], nearest=out["points"], nearest_cnt=out["cnt"])

    # --- the tape
    def _call(self, method, args, run):
        i, key = self.n, f"{self.n}.{method}."
        self.n += 1
        digest = f"{method}:{_digest(args)}"
        if self.live is not None:
            given = np.concatenate(self.given)
            for k, v in run().items():
                self.rec[key + k] = self._encode(k, np.asarray(v), given)
            self.args.append(digest)
            os.makedirs(RECORD_DIR, exist_ok=True)
            np.savez_compressed(os.path.join(RECORD_DIR, self.name + ".npz"), args=np.array(self.args), **self.rec)
        elif i >= len(self.tape["args"]) or str(self.tape["args"][i]) != digest:
            raise AssertionError(f"tape {self.name}: call {i} ({method}) was not recorded with these arguments")
        tape, names = (self.rec, list(self.rec)) if self.live is not None else (self.tape, self.tape.files)
        given = np.concatenate(self.given)
        return {f[len(key):]: self._decode(f[len(key):], tape[f], given) for f in names if f.startswith(key)}

    @staticmethod
    def _encode(kind, v, given):
        if kind not in ("rows", "points"):
            return v
        index = {}
        for i, row in enumerate(given):
            index.setdefault(row.tobytes(), i)
        flat = v.reshape(-1, 4)
        idx = np.array([index.get(r.tobytes(), -1) for r in flat], dtype=np.int64)
        assert ((idx >= 0) | ~flat.any(axis=1)).all(), "the tree returned a point it was never given"
        if kind == "rows":          # a multiset of given points: how often each one is stored
            assert (idx >= 0).all(), "the tree returned a point it was never given"
            return np.bincount(idx, minlength=len(given)).astype(np.uint8)
        return (idx + 1).reshape(v.shape[:-1]).astype(np.uint16 if len(given) < 1 << 16 else np.uint32)     # 0: no point

    @staticmethod
    def _decode(kind, v, given):
        if kind == "rows":
            return np.repeat(given, v, axis=0)
        if kind == "points":
            out = np.zeros(v.shape + (4,), dtype=np.float32)
            out[v > 0] = given[v[v > 0].astype(np.int64) - 1]
            return out
        return v
