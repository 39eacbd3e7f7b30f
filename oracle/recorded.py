"""TEST INFRASTRUCTURE ONLY -- the reference's answers to the parity tests, stored, so the tests compare against the reference
on machines where oracle/_ref cannot be built (its sources are not part of this repository).

  RecordingOracle  wraps RefOracle: every call is passed through and remembered (tests/conftest.py, LMOT_RECORD_REFERENCE_CALLS);
                   it returns what the replay will return, so a test sees the same values in both
  ReplayOracle     same interface: answers each call of a test from tests/golden/reference_calls.npz

A call is stored as the method, a digest of its arguments and its results in terms of the plain-C++ restatement
(PortOracle, built everywhere): the replay runs the restatement on the same arguments and turns its results into the
reference's with the stored corrections.
  * integer and float32 results (labels, grids, boxes, track flags) are restored bit for bit: every element where the
    restatement differs is stored, and a digest of the restored bytes must match the reference's;
  * float64 results (UKF states, velocities) are restored to within REL_TOL (relative, floor 1e-3): elements where the
    restatement differs by more are stored exactly.  The tests compare these with tolerances of 1e-5 and above.
  * results the restatement cannot compute (the cluster node's side outputs) are stored as they are, or as a digest when
    larger than FULL_LIMIT bytes (ReferenceDigest).
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import tempfile

import numpy as np

from oracle import ref as oracle

REL_TOL = 1e-7
FULL_LIMIT = 16384
METHODS = ("cell_index", "ground_remove", "polar_grid", "component_clustering", "box_fitting", "cluster_outputs",
           "tracker_reset", "tracker_num_tracks", "tracker_step", "tracker_dump", "tracker_load")


def _digest(*items) -> str:
    h = hashlib.sha256()
    for x in items:
        if isinstance(x, np.ndarray):
            a = np.ascontiguousarray(x)
            h.update(f"{a.dtype.str}{a.shape}".encode())
            h.update(a.tobytes())
        else:
            h.update(repr(x).encode())
    return h.hexdigest()[:16]


def _leaves(res):
    """results -> (structure, list of ndarray leaves)"""
    if res is None:
        return "none", []
    if isinstance(res, dict):
        return ["dict", list(res.keys())], [np.asarray(v) for v in res.values()]
    if isinstance(res, tuple):
        return ["tuple", [("int" if isinstance(v, int) else "array") for v in res]], [np.asarray(v) for v in res]
    return ("int" if isinstance(res, int) else "array"), [np.asarray(res)]


def _build(struct, leaves):
    if struct == "none":
        return None
    if struct in ("int", "array"):
        return int(leaves[0]) if struct == "int" else leaves[0]
    kind, spec = struct
    if kind == "dict":
        return dict(zip(spec, leaves))
    return tuple(int(v) if s == "int" else v for s, v in zip(spec, leaves))


def _close(ref, port):
    with np.errstate(all="ignore"):
        rel = np.abs(ref - port) / np.maximum(np.maximum(np.abs(ref), np.abs(port)), 1e-3)
    return (ref == port) | (np.isnan(ref) & np.isnan(port)) | (rel <= REL_TOL)


def _exact(leaves, enc):
    """the results restored bit for bit: everything but float64 results and digests"""
    return [a for a, e in zip(leaves, enc) if e[0] != "digest" and a.dtype != np.float64]


def _call_port(port, name, args, kw):
    """The restatement's answer (tracker calls keep its state in step with the reference's), None where it has none."""
    try:
        return getattr(port, name)(*args, **kw)
    except RuntimeError:
        return None


def private_port(mode):
    """A PortOracle on its own copy of the library: its tracker state is not shared with a PortOracle the test itself uses."""
    d = tempfile.mkdtemp(prefix="lmot_port_")
    try:
        path = os.path.join(d, "liboracle_port.so")
        shutil.copy(os.path.join(oracle.HERE, "liboracle_port.so"), path)
        return oracle.PortOracle(mode, path=path)
    finally:
        shutil.rmtree(d)


def _restore(pleaves, enc, arrays, prefix):
    """the restatement's results + the stored corrections -> the reference's results"""
    leaves = []
    for j, e in enumerate(enc):
        key = f"{prefix}_{j}"
        if e[0] == "digest":
            leaves.append(ReferenceDigest(*e[1:]))
        elif e[0] == "full":
            leaves.append(arrays[key])
        else:
            a = np.array(pleaves[j])
            if e[1]:
                a.reshape(-1)[arrays[key + "_i"]] = arrays[key + "_v"]
            leaves.append(a)
    return leaves


class ReferenceDigest:
    """A large reference result kept as shape + digest: `matches(a)` is bit-exact equality with it."""

    def __init__(self, shape, dtype, digest):
        self.shape, self.dtype, self.digest = tuple(shape), np.dtype(dtype), digest

    def matches(self, a) -> bool:
        a = np.asarray(a)
        return a.shape == self.shape and _digest(np.ascontiguousarray(a, self.dtype)) == self.digest


class RecordingOracle:
    def __init__(self, mode: str, port):
        self.ref, self.port, self.mode, self.calls, self.arrays = oracle.RefOracle(mode), port, mode, [], {}

    def __getattr__(self, name):
        if name not in METHODS:
            raise AttributeError(name)

        def call(*args, **kw):
            res = getattr(self.ref, name)(*args, **kw)
            pres = _call_port(self.port, name, args, kw)
            struct, leaves = _leaves(res)
            pleaves = _leaves(pres)[1] if pres is not None else None
            enc = []
            for j, a in enumerate(leaves):
                key = f"c{len(self.calls)}_{j}"
                p = pleaves[j] if pleaves is not None else None
                if p is None or p.shape != a.shape or p.dtype != a.dtype:
                    if a.nbytes > FULL_LIMIT:
                        enc.append(["digest", list(a.shape), a.dtype.str, _digest(a)])
                    else:
                        enc.append(["full"])
                        self.arrays[key] = a
                    continue
                if a.dtype == np.float64:
                    bad = ~_close(a, p)
                else:
                    u = f"u{a.dtype.itemsize}"
                    bad = np.ascontiguousarray(a).view(u) != np.ascontiguousarray(p).view(u)
                idx = np.flatnonzero(bad)
                if len(idx):
                    self.arrays[key + "_i"] = idx.astype(np.int64)
                    self.arrays[key + "_v"] = a.reshape(-1)[idx]
                enc.append(["port", len(idx)])
            self.calls.append([name, _digest(name, *args, *sorted(kw.items())), struct, enc, _digest(*_exact(leaves, enc))])
            # hand the test what a replay will hand it (float64 results within REL_TOL), so both see the same arguments next
            restored = _restore(pleaves, enc, self.arrays, f"c{len(self.calls) - 1}")
            return _build(struct, restored)
        return call


class ReplayOracle:
    def __init__(self, mode: str, port, calls: list, arrays, sid: int):
        self.port, self.mode, self.calls, self.arrays, self.sid, self.n = port, mode, calls, arrays, sid, 0

    def __getattr__(self, name):
        if name not in METHODS:
            raise AttributeError(name)

        def call(*args, **kw):
            i = self.n
            assert i < len(self.calls), f"{name}: call {i} of this test was not recorded from the reference"
            rname, dig_in, struct, enc, dig_out = self.calls[i]
            assert rname == name, f"call {i}: the reference was recorded answering {rname}, not {name}"
            assert _digest(name, *args, *sorted(kw.items())) == dig_in, f"call {i} ({name}): arguments differ from the recorded ones"
            self.n += 1
            pres = _call_port(self.port, name, args, kw)
            leaves = _restore(_leaves(pres)[1] if pres is not None else None, enc, self.arrays, f"s{self.sid}_c{i}")
            assert _digest(*_exact(leaves, enc)) == dig_out, f"call {i} ({name}): restored results are not the reference's"
            return _build(struct, leaves)
        return call


def load(path: str):
    """-> ({(test id, mode): stream index}, calls per stream, arrays)"""
    z = np.load(path)
    meta = json.loads(str(z["meta"]))
    return {tuple(k.split("|", 1)[::-1]): i for i, k in enumerate(meta["streams"])}, meta["calls"], z


def save(path: str, streams):
    """streams: {(test id, mode): RecordingOracle}"""
    meta, arrays = {"streams": [], "calls": []}, {}
    for sid, ((test_id, mode), rec) in enumerate(sorted(streams.items())):
        meta["streams"].append(f"{mode}|{test_id}")
        meta["calls"].append(rec.calls)
        for k, v in rec.arrays.items():
            arrays[f"s{sid}_{k}"] = v
    np.savez_compressed(path, meta=np.array(json.dumps(meta, separators=(",", ":"))), **arrays)
