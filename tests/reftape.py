"""Record / replay of the reference library's answers for tests/test_oracle_vs_reference.py.

The reference (oracle/_ref/liblkref.so, see oracle/lkref.py) can only be built where its sources are. Each test there
talks to it through `Tape`, which has the surface of the lkref module (Reference, calc_body_cov, init_plane, boxminus):

  live    the library is available: every call goes through to it; with LKREF_TAPE=record the answers are also
          written to tests/golden/ref_tape/<test>.npz (tests/golden/make_ref_golden.py does that)
  replay  the library is not available (or LKREF_TAPE=replay): every call is answered from that file, so the oracle is
          held to the reference's own numbers on any machine

Every call also stores a fingerprint of its inputs (size, sum and sum of magnitudes of each array); a replayed call
whose inputs do not match the recorded ones fails rather than answer for other inputs.

What is stored is shrunk where a full copy would be large; a replayed answer then carries less than a live one:
  map_export()   a RefMap: mapcmp.summary() of the map (a hash of every node's structure and a seeded sample of plane
                 records) in both modes, and the whole export live; tests compare it through mapcmp.compare_maps
  process()      "body" is the input cloud reordered: stored as the permutation
  get_filter()   the covariance: exact when diagonal, else quantised to COV_STEP of its largest magnitude
  world clouds   above WORLD_ROWS rows, a seeded sample of WORLD_ROWS rows; the other rows replay as NaN, so tests
                 compare the rows kept_rows() names
Arrays are kept lossless otherwise (8-byte values shuffled by significance before compression).
"""
import ast
import json
import os
import re

import numpy as np

import lkref
import mapcmp
from legkilo_b200 import abi

TAPE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_tape")
WORLD_ROWS = 64
COV_STEP = 2.0 ** -44  # of the largest magnitude: the tests hold covariances to 1e-10 of it


def mode():
    m = os.environ.get("LKREF_TAPE", "")
    if m in ("record", "replay"):
        return m
    return "live" if lkref.available() else "replay"


def tape_path(test_name):
    return os.path.join(TAPE_DIR, re.sub(r"[^A-Za-z0-9_.-]+", "_", test_name).strip("_") + ".npz")


def kept_rows(world):
    """Rows of a reference world cloud that carry values (all of them, except in a replayed sampled cloud)."""
    return ~np.isnan(world[:, 0])


class RefMap:
    """A reference map export: its mapcmp.summary(), and the whole export where the reference library ran."""

    def __init__(self, summary, blob=None):
        self.summary = summary
        self.blob = blob


def _fingerprint(args):
    fp = []

    def add(a):
        if a is None or isinstance(a, str):
            fp.append(-1.0)
        elif isinstance(a, dict):
            for k in sorted(a):
                add(a[k])
        else:
            a = np.asarray(a)
            if a.dtype.names:
                for k in a.dtype.names:
                    add(a[k])
                return
            a = a.astype(np.float64).ravel()
            fp.extend([float(a.size), float(a.sum()), float(np.abs(a).sum())])

    for a in args:
        add(a)
    return fp


class _Buf:
    """Arrays packed into one byte buffer; 8-byte values byte-shuffled (most significant bytes together)."""

    def __init__(self, data=b""):
        self.parts, self.size, self.data = [], 0, data

    def put(self, a):
        a = np.ascontiguousarray(a)
        raw = a.view(np.uint8).reshape(-1)
        shuf = a.dtype.itemsize == 8 and not a.dtype.names
        if shuf:
            raw = raw.reshape(-1, 8).T.reshape(-1)
        self.parts.append(raw.tobytes())
        ref = [self.size, raw.size, repr(np.lib.format.dtype_to_descr(a.dtype)), list(a.shape), shuf]
        self.size += raw.size
        return ref

    def get(self, ref):
        off, n, descr, shape, shuf = ref
        raw = np.frombuffer(self.data, np.uint8, n, off)
        if shuf:
            raw = raw.reshape(8, -1).T.reshape(-1)
        return raw.copy().view(np.lib.format.descr_to_dtype(ast.literal_eval(descr))).reshape(shape)


def _encode(out, buf):
    if out is None or isinstance(out, (bool, np.bool_, str)):
        return out if not isinstance(out, np.bool_) else bool(out)
    if isinstance(out, (int, np.integer)):
        return int(out)
    if isinstance(out, float):
        return {"f": out}
    if isinstance(out, np.ndarray):
        return {"a": buf.put(out)}
    if isinstance(out, RefMap):
        return {"map": {k: _encode(v, buf) for k, v in out.summary.items()}}
    if isinstance(out, tuple):
        return {"t": [_encode(v, buf) for v in out]}
    if isinstance(out, dict):
        return {"d": {k: _encode(v, buf) for k, v in out.items()}}
    raise TypeError(type(out))


def _decode(e, buf):
    if not isinstance(e, dict):
        return e
    (k, v), = e.items()
    if k == "f":
        return float(v)
    if k == "a":
        return buf.get(v)
    if k == "map":
        return RefMap({kk: _decode(vv, buf) for kk, vv in v.items()})
    if k == "t":
        return tuple(_decode(x, buf) for x in v)
    return {kk: _decode(vv, buf) for kk, vv in v.items()}


class Tape:
    def __init__(self, test_name):
        self.mode = mode()
        self.path = tape_path(test_name)
        self.calls, self.buf, self.i = [], _Buf(), 0
        if self.mode == "replay":
            with np.load(self.path) as f:
                self.calls = json.loads(f["calls"].tobytes().decode())
                self.buf = _Buf(f["buf"].tobytes())
        self.Reference = lambda *a, **kw: _Ref(self, *a, **kw)

    def call(self, name, fn, args, shrink=None, expand=None):
        """fn() answers live; shrink(answer) is what is stored, expand(stored) what a replay answers."""
        fp = _fingerprint(args)
        if self.mode == "replay":
            assert self.i < len(self.calls), f"{self.path}: more reference calls than recorded"
            rec = self.calls[self.i]
            assert rec["name"] == name, (self.path, self.i, rec["name"], name)
            np.testing.assert_allclose(fp, rec["fp"], rtol=1e-6, atol=1e-9,
                                       err_msg=f"{self.path}: inputs of call {self.i} ({name}) differ from the recorded ones")
            out = _decode(rec["out"], self.buf)
            if expand is not None:
                out = expand(out)
        else:
            out = fn()
            self.calls.append(dict(name=name, fp=fp, out=_encode(shrink(out) if shrink else out, self.buf)))
        self.i += 1
        return out

    def close(self):
        if self.mode == "replay":
            assert self.i == len(self.calls), f"{self.path}: {len(self.calls) - self.i} recorded reference calls not made"
        elif self.mode == "record":
            os.makedirs(TAPE_DIR, exist_ok=True)
            np.savez_compressed(self.path, calls=np.frombuffer(json.dumps(self.calls).encode(), np.uint8),
                                buf=np.frombuffer(b"".join(self.buf.parts), np.uint8))

    def calc_body_cov(self, pb, range_inc, degree_inc):
        return self.call("calc_body_cov", lambda: lkref.calc_body_cov(pb, range_inc, degree_inc), (pb, range_inc, degree_inc))

    def init_plane(self, pw, var, planer_threshold=0.01):
        return self.call("init_plane", lambda: lkref.init_plane(pw, var, planer_threshold), (pw, var, planer_threshold))

    def boxminus(self, a, b):
        return self.call("boxminus", lambda: lkref.boxminus(a, b), (a, b))


def _sample_world(out):
    w = out["world"]
    if len(w) <= WORLD_ROWS:
        return out
    rows = np.sort(np.random.default_rng(len(w)).choice(len(w), WORLD_ROWS, replace=False)).astype(np.int32)
    return dict(out, world=w[rows], world_rows=rows, world_len=len(w))


def _unsample_world(out):
    if "world_rows" not in out:
        return out
    out = dict(out)
    w = np.full((out.pop("world_len"), 4), np.nan, np.float32)
    w[out.pop("world_rows")] = out["world"]
    out["world"] = w
    return out


def _shrink_cov(P):
    M = P.reshape(30, 30)
    if not (M - np.diag(np.diag(M))).any():
        return dict(diag=np.diag(M).copy())
    step = np.abs(M).max() * COV_STEP
    q = np.round(M / step).astype(np.int64)
    iu = np.triu_indices(30)
    return dict(step=float(step), upper=q[iu], lower_minus_upper=q.T[iu] - q[iu])


def _expand_cov(c):
    if "diag" in c:
        return np.diag(c["diag"]).ravel()
    iu = np.triu_indices(30)
    q = np.zeros((30, 30), np.int64)
    q.T[iu] = c["upper"] + c["lower_minus_upper"]
    q[iu] = c["upper"]
    return (q * c["step"]).ravel()


class _Ref:
    """lkref.Reference through a Tape."""

    def __init__(self, tape, cfg, imu_mode_only=True, gravity=9.81, acc_norm=1.0, initialised=True):
        self.t = tape
        self.r = None if tape.mode == "replay" else lkref.Reference(cfg, imu_mode_only, gravity, acc_norm, initialised)
        tape.call("create", lambda: None, (cfg, imu_mode_only, gravity, acc_norm, initialised))

    def _do(self, name, *args, **kw):
        return self.t.call(name, lambda: getattr(self.r, name)(*args, **kw), args + tuple(kw.values()))

    def set_filter(self, x=None, P=None, Q=None, clk=None):
        self._do("set_filter", x, P, Q, clk)

    def get_filter(self):
        return self.t.call("get_filter", self.r.get_filter if self.r else None, (),
                           lambda out: (out[0], _shrink_cov(out[1])) + out[2:],
                           lambda out: (out[0], _expand_cov(out[1])) + out[2:])

    def init_process_cov(self):
        self._do("init_process_cov")

    def acc_norm(self):
        return self._do("acc_norm")

    def build_voxel_map(self, xyz_world, xyz_body, **kw):
        self._do("build_voxel_map", xyz_world, xyz_body, **kw)

    def predict_update_point(self, t, pts):
        return self.t.call("predict_update_point", lambda: self.r.predict_update_point(t, pts), (t, pts), _sample_world,
                           _unsample_world)

    def obs_imu(self, imu):
        self._do("obs_imu", imu)

    def obs_kinimu(self, kin):
        self._do("obs_kinimu", kin)

    def process(self, begin_time, end_time, pts, imu=None, kin=None):
        pts = np.ascontiguousarray(pts, np.float32)
        rows = pts.view(np.dtype((np.void, 16))).ravel()

        def shrink(out):
            order = np.argsort(rows, kind="stable")
            perm = order[np.searchsorted(rows[order], out["body"].view(rows.dtype).ravel())].astype(np.int32)
            assert np.array_equal(pts[perm], out["body"]), "process() no longer returns a reordering of its input"
            return _sample_world(dict(out, body=np.diff(perm, prepend=0)))

        def expand(out):
            return dict(_unsample_world(out), body=pts[np.cumsum(out["body"])])

        return self.t.call("process", lambda: self.r.process(begin_time, end_time, pts, imu=imu, kin=kin),
                           (begin_time, end_time, pts, imu, kin), shrink, expand)

    def map_slide(self, position_last):
        return self._do("map_slide", position_last)

    def map_export(self):
        def export():
            blob = self.r.map_export()
            return RefMap(mapcmp.summary(blob), blob)

        return self.t.call("map_export", export, ())

    def root_keys(self):
        """Keys of the map's root voxels (lk_map root table order)."""
        return self.t.call("root_keys", lambda: abi.parse_map_blob(self.r.map_export())[1]["key"].copy(), ())

    def num_roots(self):
        return self._do("num_roots")
