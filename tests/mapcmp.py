"""Structural comparison of two lk_map blobs (oracle export vs device download)."""
import hashlib

import numpy as np

from legkilo_b200 import abi


def _canon_plane(node):
    n = node["normal"].copy(); d = float(node["d"]); pv = np.zeros((6, 6))
    iu = np.triu_indices(6)
    pv[iu] = node["plane_var"]; pv = pv + np.triu(pv, 1).T
    k = int(np.argmax(np.abs(n)))
    if n[k] < 0:
        n = -n; d = -d
        pv[:3, 3:] *= -1; pv[3:, :3] *= -1
    return n, d, pv


def compare_blobs(blob_a, blob_b, rtol=1e-6, check_points=True, pt_atol=1e-12, var_rtol=1e-9, plane_tol=None):
    """blob_a: reference (oracle), blob_b: device. Returns dict of counts; raises AssertionError on mismatch.
    plane_tol(node, aux, points) -> dict(normal=, plane_var=, d=, radius=), if given, replaces the fixed plane-parameter
    tolerances (normal and d absolute, plane_var relative to its largest entry, radius relative) plane by plane; the
    largest error / tolerance ratio of each parameter is then returned in stats["ratio"]."""
    ha, ra, na, aa, pa = abi.parse_map_blob(blob_a)
    hb, rb, nb, ab, pb = abi.parse_map_blob(blob_b)
    assert int(ha["n_roots"]) == int(hb["n_roots"]), (ha["n_roots"], hb["n_roots"])
    ka = {tuple(r["key"]): int(r["node"]) for r in ra}
    kb = {tuple(r["key"]): int(r["node"]) for r in rb}
    assert set(ka) == set(kb)
    stats = dict(nodes=0, planes=0, points=0, interior=0, max_plane_err=0.0,
                 ratio=dict(normal=0.0, plane_var=0.0, d=0.0, radius=0.0))

    def cmp_node(ia, ib, path):
        A, B, XA, XB = na[ia], nb[ib], aa[ia], ab[ib]
        fa, fb = int(A["flags"]), int(B["flags"])
        stats["nodes"] += 1
        msg = f"node {path}"
        assert (fa & 0xff07) == (fb & 0xff07), (msg, hex(fa), hex(fb))  # plane/init/update + layer
        assert ((fa >> 16) & 0xff) == ((fb >> 16) & 0xff), (msg, "childmask", hex(fa), hex(fb))
        np.testing.assert_allclose(XB["voxel_center"], XA["voxel_center"], rtol=0, atol=1e-12, err_msg=msg)
        assert float(XA["quater_length"]) == float(XB["quater_length"]), msg
        layer = (fa >> 8) & 0xff
        interior = bool(fa & 2) and not (fa & 1) and ((fa >> 16) & 0xff)
        if fa & 1:
            stats["planes"] += 1
            n1, d1, p1 = _canon_plane(A); n2, d2, p2 = _canon_plane(B)
            np.testing.assert_allclose(B["center"], A["center"], rtol=0, atol=max(pt_atol, 1e-12), err_msg=msg)
            ra, rb = float(A["radius"]), float(B["radius"])
            err = dict(normal=float(np.abs(n2 - n1).max()), d=abs(d2 - d1),
                       plane_var=float(np.abs(p2 - p1).max() / np.abs(p1).max()), radius=abs(rb - ra) / max(ra, 1e-30))
            if plane_tol is None:
                tol = dict(normal=rtol, d=1e-5 * max(1.0, abs(d1)), plane_var=rtol, radius=1e-6 * max(1.0, ra) / max(ra, 1e-30))
            else:
                c = int(XA["pts_count"])
                tol = plane_tol(A, XA, pa[int(XA["pts_base"]):int(XA["pts_base"]) + c])
            for k in err:
                strict = plane_tol is None and k == "plane_var"
                assert err[k] < tol[k] if strict else err[k] <= tol[k], (msg, k, err[k], tol[k])
                stats["ratio"][k] = max(stats["ratio"][k], err[k] / tol[k] if tol[k] > 0 else 0.0)
            stats["max_plane_err"] = max(stats["max_plane_err"], err["plane_var"])
        if not interior:
            assert int(XA["pts_count"]) == int(XB["pts_count"]), (msg, "pts_count", XA["pts_count"], XB["pts_count"])
            assert int(XA["new_points"]) == int(XB["new_points"]), (msg, "new_points", XA["new_points"], XB["new_points"])
            c = int(XA["pts_count"])
            if check_points and c:
                qa = pa[int(XA["pts_base"]):int(XA["pts_base"]) + c]; qb = pb[int(XB["pts_base"]):int(XB["pts_base"]) + c]
                np.testing.assert_allclose(qb["pw"], qa["pw"], rtol=0, atol=pt_atol, err_msg=msg)
                np.testing.assert_allclose(qb["var"], qa["var"], rtol=var_rtol, atol=var_rtol * float(np.abs(qa["var"]).max()), err_msg=msg)
                stats["points"] += c
        else:
            stats["interior"] += 1
        mask = (fa >> 16) & 0xff
        for c in range(8):
            if mask & (1 << c):
                cmp_node(int(A["child_base"]) + c, int(B["child_base"]) + c, path + (c,))

    for key in sorted(ka):
        cmp_node(ka[key], kb[key], (key,))
    return stats


DIGEST_DTYPE = np.dtype([("flags", "u4"), ("pts_count", "i4"), ("new_points", "i4"), ("key", "i4", (3,)), ("center", "f8", (3,)),
                         ("normal", "f8", (3,)), ("d", "f8"), ("radius", "f8"), ("var_nn", "f8"), ("var_cc", "f8")])


def digest(blob):
    """A compact, order-canonical summary of a map blob for committed fixtures: one record per octree node in depth-first
    order (roots by ascending key, children by octant), sign-canonical plane, and the traces of the two diagonal blocks
    of plane_var (both invariant under the normal's sign)."""
    _, roots, nodes, aux, _ = abi.parse_map_blob(blob)
    out = []

    def walk(i, key):
        A, X = nodes[i], aux[i]
        f = int(A["flags"])
        rec = np.zeros(1, DIGEST_DTYPE)
        rec["flags"] = f & 0x00ffff07
        rec["key"] = key
        interior = bool(f & 2) and not (f & 1) and ((f >> 16) & 0xff)
        if not interior:
            rec["pts_count"] = X["pts_count"]; rec["new_points"] = X["new_points"]
        if f & 1:
            n, d, pv = _canon_plane(A)
            rec["center"] = A["center"]; rec["normal"] = n; rec["d"] = d; rec["radius"] = A["radius"]
            rec["var_nn"] = np.trace(pv[:3, :3]); rec["var_cc"] = np.trace(pv[3:, 3:])
        out.append(rec)
        for c in range(8):
            if (f >> 16) & (1 << c):
                walk(int(A["child_base"]) + c, key)

    for r in sorted(roots, key=lambda r: tuple(r["key"])):
        walk(int(r["node"]), r["key"])
    return np.concatenate(out) if out else np.zeros(0, DIGEST_DTYPE)


def _compare_planes(dg, dig_ref, rtol, center_atol):
    pl = (dig_ref["flags"] & 1).astype(bool)
    np.testing.assert_allclose(dg["center"][pl], dig_ref["center"][pl], rtol=0, atol=center_atol)
    np.testing.assert_allclose(dg["normal"][pl], dig_ref["normal"][pl], rtol=0, atol=rtol)
    np.testing.assert_allclose(dg["d"][pl], dig_ref["d"][pl], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(dg["radius"][pl], dig_ref["radius"][pl], rtol=1e-6)
    np.testing.assert_allclose(dg["var_nn"][pl], dig_ref["var_nn"][pl], rtol=rtol)
    np.testing.assert_allclose(dg["var_cc"][pl], dig_ref["var_cc"][pl], rtol=rtol)


def _stats(dg):
    f = dg["flags"]
    interior = ((f & 2) != 0) & ((f & 1) == 0) & (((f >> 16) & 0xff) != 0)
    return dict(nodes=len(dg), planes=int((f & 1).sum()), interior=int(interior.sum()), points=int(dg["pts_count"][~interior].sum()))


def compare_digest(dig_ref, blob, rtol=1e-6, center_atol=1e-10):
    """dig_ref: digest() of the reference's map (a committed fixture); blob: the map under test."""
    dg = digest(blob)
    assert len(dg) == len(dig_ref), (len(dg), len(dig_ref))
    np.testing.assert_array_equal(dg["key"], dig_ref["key"])
    np.testing.assert_array_equal(dg["flags"], dig_ref["flags"])
    np.testing.assert_array_equal(dg["pts_count"], dig_ref["pts_count"])
    np.testing.assert_array_equal(dg["new_points"], dig_ref["new_points"])
    _compare_planes(dg, dig_ref, rtol, center_atol)
    return _stats(dg)


SUMMARY_PLANES = 16


def _structure_hash(dg):
    h = hashlib.sha256()
    for k in ("key", "flags", "pts_count", "new_points"):
        h.update(np.ascontiguousarray(dg[k], "<i8").tobytes())
    return h.hexdigest()


def summary(blob):
    """digest() shrunk for fixtures: the node count, a hash of every node's structure (root key, flags, point counts) and
    the digest records of a seeded sample of SUMMARY_PLANES plane nodes."""
    dg = digest(blob)
    planes = np.flatnonzero(dg["flags"] & 1)
    idx = np.sort(np.random.default_rng(len(dg)).choice(planes, min(SUMMARY_PLANES, len(planes)), replace=False))
    return dict(nodes=len(dg), structure=_structure_hash(dg), sample_idx=idx.astype(np.int32), sample=dg[idx])


def compare_summary(summ, blob, rtol=1e-6, center_atol=1e-10):
    """summ: summary() of the reference's map; blob: the map under test. Structure exactly, sampled planes to tolerance."""
    dg = digest(blob)
    assert len(dg) == summ["nodes"], (len(dg), summ["nodes"])
    assert _structure_hash(dg) == summ["structure"], "map structure (root keys, node flags, point counts) differs from the reference's"
    _compare_planes(dg[summ["sample_idx"]], summ["sample"], rtol, center_atol)
    return _stats(dg)


def compare_maps(ref, blob, rtol=1e-6, pt_atol=1e-12, var_rtol=1e-9):
    """ref: a reference map as tests/reftape.py hands it out; blob: the map under test. Node by node and point by point
    with compare_blobs where the reference's whole export is at hand, against its summary always."""
    st = compare_summary(ref.summary, blob, rtol=rtol, center_atol=max(pt_atol, 1e-12))
    if ref.blob is not None:
        st = compare_blobs(ref.blob, blob, rtol=rtol, pt_atol=pt_atol, var_rtol=var_rtol)
    return st
