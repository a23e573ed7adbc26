"""The residual pass chunk by chunk against the CPU oracle's rows.

Every residual kernel except the persistent per-scan one writes one 32-double partial row per chunk (lk_device.cuh:
A = sum h^T h / R upper triangle row-major (21) | b = sum h z / R (6) | sum R | count), which the per-scan solve then
adds up. Those rows are read back here and compared, term by term, with the oracle's per-point rows summed in extended
precision over the same chunk. A per-row error of 1e-3 moves the solved state by less than 1e-5, so state-level checks
cannot see what this sees.

Covered: the throughput family (k_residual_stream2 on the hot plane images + k_residual_fallback, lk_stream2.cu) and
the latency kernel (k_residual, fused = 0, batch of one); axis-aligned, oblique and far-from-origin planes; maps from
lk_map_upload, from lk_map_build and from the incremental insert; and the dispatch configurations around them (one scan
above LATENCY_MAX_BUCKET, a streaming batch with ragged bucket counts, sub-ranges of one staged batch)."""
import numpy as np
import pytest

import lko
import mapcmp
import scenes
from legkilo_b200 import Engine, abi, synth

pytestmark = pytest.mark.gpu

TOL = 1e-5       # state / covariance (BASELINE.json north_star)
TERM_TOL = 1e-9  # per chunk and term, relative to the sum of |contributions| (the debug-row tests' row tolerance)
# z = -(float)(n . pw + d) on both sides (voxel_map.cc:658, a float dis_to_plane_). pw itself is formed in double with a
# different operation order on the device, so far from the origin (|pw| ~ 1e4 m against |z| ~ 1e-2 m, pw differing by
# ~eps |pw|) the float rounding of z can go the other way on a few rows. Far away only (|x0.pos| > FAR_M), b = sum h z / R
# may also differ by one float ulp of z on at most MAX_Z_FLIPS rows of a chunk: the largest such contributions.
FAR_M = 100.0
MAX_Z_FLIPS = 4

# ---- the chunk model: lk_api.cu chunk_size_for / build_tables -------------------------------------------------------
LATENCY_MAX_BUCKET = 148 * 256  # one 256-point chunk per SM of a B200: the per-scan kernel's reach
SMALL_CHUNK, BIG_CHUNK = 256, 3840
NACC = 29  # A (21) | b (6) | sum R | count
ACC_B, ACC_SUMR, ACC_CNT = 21, 27, 28


def chunk_size(n, n_scans):
    """Points per chunk of a bucket of n points in a call with n_scans scans (chunk_size_for)."""
    if n_scans >= 2:
        return SMALL_CHUNK if n <= 2048 else BIG_CHUNK
    return SMALL_CHUNK if n <= LATENCY_MAX_BUCKET else BIG_CHUNK


def chunk_table(scan_bucket_ptr, bucket_offsets):
    """build_tables: [(scan, first point, count)] step-major (bucket rank k), then scan, then consecutive chunks of
    the bucket. Empty buckets have no chunk."""
    sbp = [int(v) for v in scan_bucket_ptr]
    bo = [int(v) for v in bucket_offsets]
    batch = len(sbp) - 1
    nb = [sbp[s + 1] - sbp[s] for s in range(batch)]
    out = []
    for k in range(max(nb, default=0)):
        for s in range(batch):
            if k >= nb[s]:
                continue
            p0, p1 = bo[sbp[s] + k], bo[sbp[s] + k + 1]
            cs = chunk_size(p1 - p0, batch)
            out += [(s, q, min(cs, p1 - q)) for q in range(p0, p1, cs)]
    return out


def one_bucket_per_scan(scan_offsets):
    return np.arange(len(scan_offsets), dtype=np.uint32), np.asarray(scan_offsets, np.uint32)


# ---- the oracle's side ----------------------------------------------------------------------------------------------
def row_terms(ok, h, z, R):
    """The 29 accumulated terms of every point's row (zeros where no row): accumulate_row's layout."""
    ok = np.asarray(ok).astype(bool)
    t = np.zeros((len(ok), NACC))
    w = np.zeros(len(ok))
    w[ok] = 1.0 / R[ok]
    r, c = np.triu_indices(6)  # row-major r <= c, accumulate_row's order
    t[:, :21] = h[:, r] * h[:, c] * w[:, None]
    t[:, ACC_B:ACC_B + 6] = h * (z * w)[:, None]
    t[:, ACC_SUMR] = np.where(ok, R, 0.0)
    t[:, ACC_CNT] = ok
    t[~ok] = 0.0
    return t


def z_slack(ok, h, z, R):
    """Per point and b term: |h / R| times one float32 ulp of |z| (what rounding z the other way moves)."""
    ok = np.asarray(ok).astype(bool)
    t = np.zeros((len(ok), NACC))
    ulp = np.spacing(np.abs(z).astype(np.float32)).astype(np.float64)
    t[ok, ACC_B:ACC_B + 6] = np.abs(h[ok]) / R[ok, None] * ulp[ok, None]
    return t


def chunk_sums(terms, chunks, scan_offsets):
    """Per chunk: the sum of its points' terms in extended precision, and the sum of their magnitudes (the scale a
    cancelling term is compared on)."""
    tot = np.zeros((len(chunks), NACC))
    mag = np.zeros((len(chunks), NACC))
    for i, (s, start, count) in enumerate(chunks):
        lo = start - int(scan_offsets[s])
        blk = terms[s][lo:lo + count].astype(np.longdouble)
        tot[i] = blk.sum(0)
        mag[i] = np.abs(blk).sum(0)
    return tot, mag


def oracle_rows(cfg, blob, pts, x0, P0, iters=1):
    """One bucket at t = 0 (no predict: both clocks 0) with the oracle's rows of the last iteration."""
    o = lko.Oracle(cfg)
    o.map_import(blob)
    o.set_filter(x0, P0, abi.process_cov_Q(cfg), np.zeros(1, abi.CLOCK_DTYPE))
    o.set_options(gain_mode=lko.GAIN_INFORMATION, iters=iters, update_map=False)
    r = o.predict_update_point(0.0, pts, debug=True)
    x, P, _, _ = o.get_filter()
    return r, x, P


def info_form_update(x0, P0, A, b):
    """ESKF::updateByPoints in information form from the summed terms: dx = (P^-1 + H^T R^-1 H)^-1 H^T R^-1 z,
    P+ = (P^-1 + H^T R^-1 H)^-1 with H = [h | 0]. Returns (x0 [+] dx, P+)."""
    P = np.asarray(P0, np.float64).reshape(30, 30)
    Am = np.zeros((6, 6))
    Am[np.triu_indices(6)] = A
    Am = Am + np.triu(Am, 1).T
    M = np.linalg.inv(P)
    M[:6, :6] += Am
    rhs = np.zeros(30)
    rhs[:6] = b
    dx = np.linalg.solve(M, rhs)
    return lko.boxplus(x0, dx), np.linalg.inv(M)


# ---- which branch of the reference a row came from ----------------------------------------------------------------
HOME, DESCENT, NEIGHBOUR = "home", "descent", "neighbour"


def classify_rows(blob, ok, h, key):
    """Per row: HOME when the home root voxel is a plane and the row's normal is +-its normal; DESCENT when the home
    root is not a plane (octree descent, voxel_map.cc:412-424); NEIGHBOUR when the home root is a plane with another
    normal (it gated the point out and the one neighbour voxel produced the row, KILO.cc:156-178)."""
    _, roots, nodes, _, _ = abi.parse_map_blob(blob)
    root_of = {tuple(int(v) for v in r["key"]): int(r["node"]) for r in roots}
    ok = np.asarray(ok).astype(bool)
    lab = np.full(len(ok), "", dtype=object)
    for i in np.flatnonzero(ok):
        nd = nodes[root_of[tuple(int(v) for v in key[i])]]
        if not int(nd["flags"]) & abi.NODE_IS_PLANE:
            lab[i] = DESCENT
            continue
        n = h[i, 3:6]
        same = min(np.abs(n - nd["normal"]).max(), np.abs(n + nd["normal"]).max()) < 1e-12
        lab[i] = HOME if same else NEIGHBOUR
    return lab


def path_counts(labels):
    return {p: int((labels == p).sum()) for p in (HOME, DESCENT, NEIGHBOUR)}


# ---- the check ------------------------------------------------------------------------------------------------------
def gate_margin(cfg, r, P0):
    """Per oracle row: |z| / (sigma_num sqrt(sigma_l)) (voxel_map.cc:387 accepts below 1), with sigma_l = R / ratio + the
    state part h_t^T P_tt h_t + n^T P_pp n; NaN where the oracle produced no row."""
    P = np.asarray(P0, np.float64).reshape(30, 30)
    h = r["h"]
    st = np.einsum("ni,ij,nj->n", h[:, :3], P[:3, :3], h[:, :3]) + np.einsum("ni,ij,nj->n", h[:, 3:], P[3:6, 3:6], h[:, 3:])
    sig = r["R"] / cfg["lidar_point_meas_ratio"] + st
    with np.errstate(divide="ignore", invalid="ignore"):
        m = np.abs(r["z"]) / (cfg["sigma_num"] * np.sqrt(sig))
    return np.where(r["ok"].astype(bool), m, np.nan)


def _explain_count(chunk, dev, ref, r, lo, dbg, margin):
    """A count mismatch: the points of the chunk whose row presence differs between the oracle and the device's latency
    debug kernel, and the oracle rows closest to the gate, each with its home key and gate margin."""
    count = chunk[2]
    ok = r["ok"][lo:lo + count].astype(bool)
    lines = [f"chunk {chunk}: device counted {dev[ACC_CNT]:.0f} rows, oracle {ref[ACC_CNT]:.0f}"]
    if dbg is not None:
        diff = np.flatnonzero(dbg["ok"].astype(bool) != ok)
        lines.append(f"row presence differs (debug kernel vs oracle) at points {(diff + lo).tolist()[:16]}, home keys "
                     f"{r['key'][lo + diff].tolist()[:16]}, oracle margins {np.round(margin[lo + diff], 6).tolist()[:16]}")
    m = margin[lo:lo + count]
    near = np.argsort(np.abs(np.nan_to_num(m, nan=np.inf) - 1.0))[:8]
    lines.append(f"oracle rows nearest the gate: points {(near + lo).tolist()}, home keys {r['key'][lo + near].tolist()}, "
                 f"margins {np.round(m[near], 6).tolist()}, rows without a row in the chunk {int((~ok).sum())}")
    return "; ".join(lines)


def check_partials(dev, chunks, scan_offsets, rows, label="", far=False, explain=None):
    """dev: [n_chunks, 32] device rows; rows[s]: the oracle's debug rows of scan s. Counts exact, every term within
    TERM_TOL of its chunk's magnitude (plus, far from the origin, the z rounding of MAX_Z_FLIPS rows on b). explain(s, lo,
    count) describes a count mismatch. Returns the largest relative term error."""
    assert dev.shape[0] == len(chunks)
    terms = [row_terms(r["ok"], r["h"], r["z"], r["R"]) for r in rows]
    tot, mag = chunk_sums(terms, chunks, scan_offsets)
    for i, (s, start, count) in enumerate(chunks):
        if dev[i, ACC_CNT] != tot[i, ACC_CNT]:
            lo = start - int(scan_offsets[s])
            pytest.fail(f"{label} " + (explain(chunks[i], dev[i], tot[i], s, lo) if explain else str(chunks[i])))
    slack = np.zeros((len(chunks), ACC_CNT))
    if far:
        zs = [z_slack(r["ok"], r["h"], r["z"], r["R"]) for r in rows]
        for i, (s, start, count) in enumerate(chunks):
            lo = start - int(scan_offsets[s])
            slack[i] = np.sort(zs[s][lo:lo + count, :ACC_CNT], axis=0)[-MAX_Z_FLIPS:].sum(0)
    err = np.abs(dev[:, :ACC_CNT] - tot[:, :ACC_CNT])
    scale = mag[:, :ACC_CNT]
    assert np.all(err[scale == 0] == 0), label
    rel = np.where(scale > 0, err / np.where(scale > 0, scale, 1.0), 0.0)
    bad = err > TERM_TOL * scale + slack
    if bad.any():
        i, j = np.argwhere(bad)[0]
        pytest.fail(f"{label} chunk {chunks[i]} term {j}: device {dev[i, j]!r} oracle {tot[i, j]!r} rel {rel[i, j]:.3e} "
                    f"(allowed {TERM_TOL:.0e} + float z rounding {slack[i, j] / max(scale[i, j], 1e-300):.1e})")
    return float(rel.max()) if rel.size else 0.0


def run_family(cfg, blob, scans, x0, family, eng=None, min_paths=None, label=""):
    """Stage the scans (one bucket each, t = 0, no predict), run one iteration through `family` ("throughput": all
    scans in one call; "latency": each scan alone with fused = 0), read the partial rows back and hold them to the
    oracle's. Also checks n_eff exactly and the state / covariance to TOL. Returns (max term error, path counts)."""
    B = len(scans)
    x0 = np.asarray(x0, abi.STATE_DTYPE)
    if len(x0) == 1 and B > 1:
        x0 = np.repeat(x0, B)
    P0 = abi.init_cov(B)
    Q = abi.process_cov_Q(cfg)
    if eng is None:
        eng = Engine(cfg)
        eng.map_upload(blob)
    rows, xs, Ps = [], [], []
    for i, s in enumerate(scans):
        r, xo, Po = oracle_rows(cfg, blob, s, x0[i:i + 1], P0[i:i + 1])
        rows.append(r); xs.append(xo); Ps.append(Po)
    far = float(np.abs(x0["pos"]).max()) > FAR_M
    margins = [gate_margin(cfg, r, P0[i]) for i, r in enumerate(rows)]

    def explain(chunk, dev_row, ref_row, s, lo):
        sp = scans[s][lo:lo + chunk[2]]
        dbg = eng.debug_residuals(x0[s:s + 1], P0[s:s + 1], sp) if len(sp) else None
        return _explain_count(chunk, dev_row, ref_row, rows[s], lo, dbg, margins[s])

    counts = {HOME: 0, DESCENT: 0, NEIGHBOUR: 0}
    for r in rows:
        for k, v in path_counts(classify_rows(blob, r["ok"], r["h"], r["key"])).items():
            counts[k] += v
    worst = 0.0
    if family == "throughput":
        assert B >= 2
        pts = np.concatenate(scans)
        offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.uint32)
        out = eng.scan_update(x0, P0, Q, np.zeros(B, abi.CLOCK_DTYPE), pts, offs, np.zeros(B), iters=1, want_world=False)
        chunks = chunk_table(*one_bucket_per_scan(offs))
        dev = eng.debug_partials(len(chunks))
        worst = check_partials(dev, chunks, offs, rows, label, far, explain)
        outs = [(out, i) for i in range(B)]
    else:
        eng.set_param("fused", 0)
        outs = []
        for i, s in enumerate(scans):
            offs = np.array([0, len(s)], np.uint32)
            out = eng.scan_update(x0[i:i + 1], P0[i:i + 1], Q, np.zeros(1, abi.CLOCK_DTYPE), s, offs, [0.0], iters=1,
                                  want_world=False)
            chunks = chunk_table(*one_bucket_per_scan(offs))
            dev = eng.debug_partials(len(chunks))
            worst = max(worst, check_partials(dev, chunks, offs, rows[i:i + 1], f"{label}[{i}]", far,
                                              lambda c, d, t, s, lo, i=i: explain(c, d, t, i, lo)))
            outs.append((out, 0))
        eng.set_param("fused", 1)
    for i, (out, j) in enumerate(outs):
        assert int(out["n_eff"][j]) == rows[i]["n_eff"], (label, i)
        if rows[i]["n_eff"]:
            assert scenes.rel_state_err(out["x"][j:j + 1], xs[i], x0[i:i + 1]) < TOL, (label, i)
            assert scenes.rel_cov_err(out["P"][j], Ps[i]) < TOL, (label, i)
    print(f"\n{label} [{family}]: max term error {worst:.2e}, rows {counts}")
    for p, m in (min_paths or {}).items():
        assert counts[p] >= m, (label, family, p, counts)
    return worst, counts


# ---- scenes ---------------------------------------------------------------------------------------------------------
EDGE_SIZES = (1, 31, 33, 255, 256, 257, 2047, 2048, 2049, 3839, 3840, 3841)
FAR = ((1500.0, -2500.0, 40.0), (12000.0, 8000.0, 0.0))
# rows every scene must produce, per path (the oblique scene's neighbour rows come from its split-level facets, at
# every offset: see scenes.OBLIQUE_FACETS)
MIN_BOX = {HOME: 20000}
MIN_OBLIQUE = {HOME: 10000, DESCENT: 1000, NEIGHBOUR: 6}
MIN_OBLIQUE_ONE = {HOME: 5000, DESCENT: 500, NEIGHBOUR: 2}  # one scan of the two


def edge_pieces(scan):
    """Consecutive slices of one scan with the chunk-edge lengths of the throughput family: one point, group (32) and
    chunk (256 / 3 840) boundaries +-1, and the 2 048 / 2 049 switch between 256- and 3 840-point chunks."""
    out, o = [], 0
    for n in EDGE_SIZES:
        assert o + n <= len(scan)
        out.append(scan[o:o + n].copy())
        o += n
    return out


def _box(offset=(0.0, 0.0, 0.0), batch=2, **kw):
    cfg, pw, pb, scans, x0 = scenes.box_points(offset=offset, batch=batch, **kw)
    return cfg, pw, pb, scans, x0


def test_box_room_chunks():
    cfg, pw, pb, scans, x0 = _box(batch=2)
    blob = scenes.oracle_map(cfg, pw, pb)
    eng = Engine(cfg)
    eng.map_upload(blob)
    run_family(cfg, blob, scans, x0, "throughput", eng, MIN_BOX, "box room")
    pieces = edge_pieces(scans[0])
    run_family(cfg, blob, pieces, x0[:1], "throughput", eng, label="box room, chunk edges")
    run_family(cfg, blob, scans[:1], x0[:1], "latency", eng, {HOME: 10000}, "box room")


def test_oblique_facets_chunks():
    cfg, pw, pb, scans, x0 = scenes.oblique_scene(batch=2, n_scan=24000)
    blob = scenes.oracle_map(cfg, pw, pb)
    eng = Engine(cfg)
    eng.map_upload(blob)
    run_family(cfg, blob, scans, x0, "throughput", eng, MIN_OBLIQUE, "oblique")
    run_family(cfg, blob, edge_pieces(scans[0]), x0[:1], "throughput", eng, label="oblique, chunk edges")
    run_family(cfg, blob, scans[:1], x0[:1], "latency", eng, MIN_OBLIQUE_ONE, "oblique")


@pytest.mark.parametrize("offset", FAR, ids=["1.5km", "12km"])
@pytest.mark.parametrize("scene", ["box", "oblique"])
def test_far_from_origin_chunks(scene, offset):
    """The reference keeps d and dis_to_plane in float: far from the origin |z| differs from n.(pw - c) by ~1e-4 m,
    which the kernels must reproduce row by row."""
    if scene == "box":
        cfg, pw, pb, scans, x0 = _box(offset=offset, batch=2)
        need, need_one = MIN_BOX, {HOME: 10000}
    else:
        cfg, pw, pb, scans, x0 = scenes.oblique_scene(offset=offset, batch=2, n_scan=24000)
        need, need_one = MIN_OBLIQUE, MIN_OBLIQUE_ONE
    blob = scenes.oracle_map(cfg, pw, pb)
    eng = Engine(cfg)
    eng.map_upload(blob)
    run_family(cfg, blob, scans, x0, "throughput", eng, need, f"{scene} at {offset}")
    run_family(cfg, blob, edge_pieces(scans[0]), x0[:1], "throughput", eng, label=f"{scene} at {offset}, chunk edges")
    run_family(cfg, blob, scans[:1], x0[:1], "latency", eng, need_one, f"{scene} at {offset}")


# ---- the other producers of the hot images --------------------------------------------------------------------------
EPS = np.finfo(np.float64).eps
NORMAL_SCALE = 4000.0  # largest normal error of a built map / (eps L^2): measured 650 (1.5 km) and 1000 (12 km)
F32_ULP = 2.0 ** -23


def plane_tol_for(cloud):
    """plane_tol over the points a map was built from (float32 world [n, 3]): a node's fit set is the cloud inside its
    cube, voxel_center +- 2 quater_length (the map keeps no points for many planes)."""
    cloud = np.asarray(cloud, np.float64)

    def tol(node, aux, _stored):
        c, h = np.asarray(aux["voxel_center"], np.float64), 2.0 * float(aux["quater_length"])
        inside = np.all((cloud >= c - h) & (cloud < c + h), axis=1)
        return plane_tol(node, cloud[inside])
    return tol


def plane_tol(node, p):
    """Plane-parameter tolerances of a map built twice from the same float32 points p (lk_map_build against the oracle).

    Both form the covariance in one pass, S = E[x x^T] - c c^T (voxel_map.cc:49-54), in double but in a different
    order (the device with fused multiply-adds). A sum of N terms of size L^2 (L = the largest |x| in the node) is off by
    at most (N - 1) eps L^2 N, so each entry of E[x x^T] by N eps L^2, c c^T by 2 N eps L^2: |dS|_2 <= 3 x 2 x 3 (N + 1)
    eps L^2 = 18 (N + 1) eps L^2 for the two implementations together. The centres agree exactly (the same sums of the
    same points), so centres and stored points are compared at 1e-12 elsewhere. The normal, the eigenvector of the
    smallest eigenvalue, moves by at most |dS| / gap (Davis-Kahan), gap = lambda_2 - lambda_1 of the node's points.
    plane_var is built from the eigenvectors and 1 / (lambda_1 - lambda_k) (voxel_map.cc:60-80): 8x the normal's bound
    relative to its largest entry. d = -n . c (a float) moves by |dn| |c| plus its own rounding, radius = sqrt(lambda_3)
    (a float) by dS / (2 lambda_3) relative plus its rounding. Floors: what a voxel near the origin reaches with two
    different 3x3 eigen-solvers. This bound is a worst case; _compare_built_maps also holds the largest normal error of
    the whole map to the measured scale law."""
    n = max(len(p), 1)
    L2 = float((p * p).sum(1).max()) if len(p) else float(np.dot(node["center"], node["center"]))
    lam = np.linalg.eigvalsh(np.cov(p.T, bias=True)) if len(p) >= 3 else np.array([0.0, 1.0, 1.0])
    gap = max(lam[1] - lam[0], 1e-12)
    dS = 18 * (n + 1) * EPS * L2
    dn = max(1e-9, dS / gap)
    return dict(normal=dn, plane_var=max(1e-8, 8 * dn),
                d=dn * float(np.linalg.norm(node["center"])) + 2 * F32_ULP * max(1.0, abs(float(node["d"]))),
                radius=max(1e-6, dS / (2 * max(lam[2], 1e-12)) + 2 * F32_ULP))


def _compare_built_maps(ref, dev, cloud, offset):
    """The whole map node by node (mapcmp.compare_blobs): structure and every stored point exact, voxel and plane
    centres to 1e-12 m, plane parameters within plane_tol. Prints the largest error / tolerance ratio per parameter."""
    st = mapcmp.compare_blobs(ref, dev, pt_atol=1e-12, var_rtol=1e-9, plane_tol=plane_tol_for(cloud))
    da, db = mapcmp.digest(ref), mapcmp.digest(dev)
    pl = (da["flags"] & 1).astype(bool)
    ne = float(np.abs(db["normal"][pl] - da["normal"][pl]).max())
    de = float(np.abs(db["d"][pl] - da["d"][pl]).max())
    ce = float(np.abs(db["center"][pl] - da["center"][pl]).max())
    print(f"\nbuilt map at {offset}: {st['planes']} planes, {st['points']} points; normal {ne:.2e}, d {de:.2e} m, "
          f"centre {ce:.2e} m, plane_var {st['max_plane_err']:.2e}; error / tolerance "
          + ", ".join(f"{k} {v:.2f}" for k, v in st["ratio"].items()))
    assert st["planes"] > 500 and st["points"] > 10000
    # the typical rounding is far below the worst case above: measured on a B200 the largest normal error of the map is
    # ~600-1000 eps L^2 (1.2e-6 at 1.5 km, 4.7e-5 at 12 km); a normal off by 1e-3, or a centre formed in float, fails
    assert ne <= max(1e-9, NORMAL_SCALE * EPS * (float(np.dot(offset, offset)) + 100.0)), ne
    return st


@pytest.mark.parametrize("offset", ((0.0, 0.0, 0.0),) + FAR, ids=["origin", "1.5km", "12km"])
def test_device_built_map_chunks(offset):
    """lk_map_build fills the hot images in node_reset / hot_after_fit: the oracle reads the device's own map, so any
    difference in the partial rows comes from the hot images, not from map numerics."""
    cfg, pw, pb, scans, x0 = scenes.oblique_scene(offset=offset, batch=2, n_scan=24000)
    eng = Engine(cfg)
    eng.map_build(pw, pb)
    dev = eng.map_download()
    _compare_built_maps(scenes.oracle_map(cfg, pw, pb), dev, pw, offset)
    run_family(cfg, dev, scans, x0, "throughput", eng, MIN_OBLIQUE, f"device-built map at {offset}")
    run_family(cfg, dev, scans[:1], x0[:1], "latency", eng, MIN_OBLIQUE_ONE, f"device-built map at {offset}")


@pytest.mark.parametrize("insert", ["two-launch", "slice-and-sort", "in-kernel"])
def test_incremental_insert_chunks(insert):
    """One streaming scan inserted with update_map (refits every few points per leaf, new roots and octants), then a
    batch of two other scans against the map it left: stale hot images would show here."""
    import test_gpu_parity as tp
    cfg, blob, scans = scenes.box_scene(batch=3, streaming=True, stream0=700)
    eng = Engine(cfg)
    eng.set_param("fast_insert", 0 if insert == "slice-and-sort" else 1)
    eng.set_param("fused_insert", 1 if insert == "in-kernel" else 0)
    eng.map_upload(blob)
    x0 = tp._moving_state(); P0 = abi.init_cov(1)
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 9.99; clk["last_update_time"] = 9.985
    pts, offs, times = synth.bucketize(scans[0], begin_time=10.0)
    eng.scan_update(x0, P0, abi.process_cov_Q(cfg), clk, pts, [0, len(pts)], times, scan_bucket_ptr=[0, len(times)],
                    bucket_offsets=offs, update_map=True)
    assert eng.map_stats()["points"] > int(abi.parse_map_blob(blob)[0]["n_points"])
    dev = eng.map_download()
    eng.set_param("fused_insert", 0)
    run_family(cfg, dev, scans[1:], abi.default_states(1), "throughput", eng, MIN_BOX, f"after insert ({insert})")


# ---- dispatch configurations ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("update_map", [False, True])
def test_one_scan_above_latency_reach(update_map):
    """An OS64 scan (> LATENCY_MAX_BUCKET points) alone in a call takes the throughput kernels on 3 840-point chunks."""
    cfg, pw, pb, scans, x0 = _box(batch=1, lidar=synth.OS64, stream0=1700)
    s = scans[0]
    assert len(s) > LATENCY_MAX_BUCKET
    blob = scenes.oracle_map(cfg, pw, pb)
    eng = Engine(cfg)
    eng.map_upload(blob)
    if not update_map:
        run_family(cfg, blob, [s], x0, "latency", eng, {HOME: 40000}, "one OS64 scan")
        return
    P0 = abi.init_cov(1)
    o = lko.Oracle(cfg)
    o.map_import(blob)
    o.set_filter(x0, P0, abi.process_cov_Q(cfg), np.zeros(1, abi.CLOCK_DTYPE))
    o.set_options(gain_mode=lko.GAIN_INFORMATION, iters=1, update_map=True)
    ro = o.predict_update_point(0.0, s)
    xo, Po, _, _ = o.get_filter()
    out = eng.scan_update(x0, P0, abi.process_cov_Q(cfg), np.zeros(1, abi.CLOCK_DTYPE), s, [0, len(s)], [0.0],
                          update_map=True)
    assert int(out["n_eff"][0]) == ro["n_eff"] > 0
    assert scenes.rel_state_err(out["x"], xo, x0) < TOL
    assert scenes.rel_cov_err(out["P"][0], Po) < TOL
    np.testing.assert_array_equal(out["world"][:, 3], ro["world"][:, 3])
    # the device state differs from the oracle's by ~1e-11 relative, so do the inserted points (as in test_gpu_map)
    st = mapcmp.compare_blobs(o.map_export(), eng.map_download(), rtol=1e-5, pt_atol=1e-8, var_rtol=1e-6)
    assert st["points"] > len(s)


def test_streaming_batch_with_ragged_bucket_counts():
    """Four streams in one call: ~50 buckets, a truncated scan with fewer buckets, a single bucket and no bucket at
    all. Steps where a scan has no bucket go through k_predict_prepare and k_scan_tail's inactive exit; every scan must
    match the oracle's own bucket loop."""
    import test_gpu_parity as tp
    cfg, blob, scans = scenes.box_scene(batch=3, streaming=True, stream0=1900)
    t0 = 10.0
    full = synth.bucketize(scans[0], begin_time=t0)
    p1, o1, _ = synth.bucketize(scans[1], begin_time=t0)
    short = synth.bucketize(p1[:o1[12]].copy(), begin_time=t0)
    single = scans[2].copy()
    single[:, 3] = 0.0
    single = synth.bucketize(single, begin_time=t0)
    empty = synth.bucketize(np.zeros((0, 4), np.float32), begin_time=t0)
    streams = [full, short, single, empty]
    nb = [len(s[2]) for s in streams]
    assert nb[0] > nb[1] > nb[2] == 1 and nb[3] == 0
    B = len(streams)
    pts = np.concatenate([s[0] for s in streams])
    so = np.concatenate([[0], np.cumsum([len(s[0]) for s in streams])]).astype(np.uint32)
    sbp = np.concatenate([[0], np.cumsum(nb)]).astype(np.uint32)
    bo = np.concatenate([[0]] + [so[i] + s[1][1:] for i, s in enumerate(streams)]).astype(np.uint32)
    bt = np.concatenate([s[2] for s in streams])
    x0 = np.repeat(tp._moving_state(), B); P0 = abi.init_cov(B)
    clk0 = np.zeros(B, abi.CLOCK_DTYPE); clk0["last_predict_time"] = 9.99; clk0["last_update_time"] = 9.985
    eng = Engine(cfg)
    eng.map_upload(blob)
    out = eng.scan_update(x0, P0, abi.process_cov_Q(cfg), clk0, pts, so, bt, scan_bucket_ptr=sbp, bucket_offsets=bo, iters=2)
    for i, (p, _, _) in enumerate(streams):
        ro, xo, Po, clko, _ = tp._oracle_stream(cfg, blob, p, t0, x0[i:i + 1], P0[i:i + 1], clk0[i:i + 1], iters=2)
        assert int(out["n_eff"][i]) == ro["n_eff"], i
        if len(p):
            assert ro["n_eff"] > 0
            assert scenes.rel_state_err(out["x"][i:i + 1], xo, x0[i:i + 1]) < TOL, i
            assert scenes.rel_cov_err(out["P"][i], Po) < TOL, i
        else:
            assert out["x"][i:i + 1].tobytes() == x0[i:i + 1].tobytes()
            np.testing.assert_array_equal(out["P"][i], P0[i])
        assert out["clk"][i].tobytes() == clko[0].tobytes(), (i, out["clk"][i], clko[0])
        np.testing.assert_array_equal(out["world"][so[i]:so[i + 1], 3], ro["world"][:, 3], err_msg=str(i))


def test_sub_ranges_of_one_staged_batch_are_bitwise_equal():
    """run_range over [0, k) and then [k, B) computes what one run_range(0, B) computes, bit for bit."""
    cfg, blob, scans = scenes.box_scene(batch=5, stream0=2300)
    B, k = len(scans), 2
    pts = np.concatenate(scans)
    so = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.uint32)
    x0 = abi.default_states(B); P0 = abi.init_cov(B); clk = np.zeros(B, abi.CLOCK_DTYPE); Q = abi.process_cov_Q(cfg)
    eng = Engine(cfg)
    eng.map_upload(blob)
    eng.stage(x0, P0, Q, clk, pts, so, np.zeros(B))
    eng.run_range(0, B, iters=2)
    eng.sync()
    whole = eng.fetch(want_world=False)
    eng.stage(x0, P0, Q, clk, pts, so, np.zeros(B))
    eng.run_range(0, k, iters=2)
    eng.run_range(k, B - k, iters=2)
    eng.sync()
    parts = eng.fetch(want_world=False)
    assert whole["n_eff"].min() > 0
    assert parts["x"].tobytes() == whole["x"].tobytes()
    assert parts["P"].tobytes() == whole["P"].tobytes()
    np.testing.assert_array_equal(parts["n_eff"], whole["n_eff"])
