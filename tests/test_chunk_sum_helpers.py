"""CPU checks of the helpers behind tests/test_gpu_chunk_sums.py: the chunk model, the per-chunk term sums and the
path classifier, against the CPU oracle alone."""
import numpy as np
import pytest

import mapcmp
import scenes
import test_gpu_chunk_sums as cs
from legkilo_b200 import abi


def test_chunk_model_hand_worked_cases():
    # one scan per call: 256-point chunks up to 148 x 256 = 37 888 points, then 3 840
    assert cs.chunk_size(1, 1) == 256 and cs.chunk_size(37888, 1) == 256 and cs.chunk_size(37889, 1) == 3840
    # >= 2 scans per call: 256 up to 2 048, then 3 840
    assert cs.chunk_size(2048, 2) == 256 and cs.chunk_size(2049, 2) == 3840 and cs.chunk_size(37888, 3) == 3840
    assert cs.chunk_table([0, 1], [0, 37888]) == [(0, 256 * i, 256) for i in range(148)]
    assert cs.chunk_table([0, 1], [0, 37889]) == [(0, 3840 * i, 3840) for i in range(9)] + [(0, 34560, 3329)]
    # two scans of 2 048 and 2 049 points, one bucket each
    assert cs.chunk_table([0, 1, 2], [0, 2048, 4097]) == [(0, 256 * i, 256) for i in range(8)] + [(1, 2048, 2049)]
    # step-major: bucket rank 0 of every scan, then rank 1; an empty bucket has no chunk, a scan without buckets none
    sbp = [0, 2, 2, 3]
    bo = [0, 300, 300, 310]
    assert cs.chunk_table(sbp, bo) == [(0, 0, 256), (0, 256, 44), (2, 300, 10)]
    sbp = [0, 3, 4]
    bo = [0, 10, 2059, 2060, 2070]
    assert cs.chunk_table(sbp, bo) == [(0, 0, 10), (1, 2060, 10), (0, 10, 2049), (0, 2059, 1)]


def test_chunk_sums_reproduce_the_oracle_update():
    """The summed A and b of every chunk, fed to an information-form update in numpy, give the oracle's one-iteration
    state and covariance: the term layout and order the device rows are compared in are the filter's."""
    cfg, blob, scans = scenes.box_scene(batch=1, stream0=300)
    pts = scans[0]
    x0 = abi.default_states(1); P0 = abi.init_cov(1)
    r, xo, Po = cs.oracle_rows(cfg, blob, pts, x0, P0)
    offs = np.array([0, len(pts)], np.uint32)
    chunks = cs.chunk_table(*cs.one_bucket_per_scan(offs))
    assert len(chunks) == (len(pts) + 255) // 256
    tot, mag = cs.chunk_sums([cs.row_terms(r["ok"], r["h"], r["z"], r["R"])], chunks, offs)
    assert tot[:, cs.ACC_CNT].sum() == r["n_eff"] > 0
    assert np.all(mag[:, cs.ACC_SUMR] == tot[:, cs.ACC_SUMR])
    A = tot[:, :21].sum(0)
    b = tot[:, cs.ACC_B:cs.ACC_B + 6].sum(0)
    x, P = cs.info_form_update(x0, P0, A, b)
    assert scenes.rel_state_err(x, xo, x0) < 1e-9
    assert scenes.rel_cov_err(P, Po) < 1e-9
    # and a wrong layout would not: b with two terms swapped
    bs = b.copy(); bs[[0, 3]] = bs[[3, 0]]
    assert scenes.rel_state_err(cs.info_form_update(x0, P0, A, bs)[0], xo, x0) > 1e-3


def test_path_classifier_reaches_each_scenes_paths():
    cfg, pw, pb, scans, x0 = scenes.box_points(batch=1)
    blob = scenes.oracle_map(cfg, pw, pb)
    r, _, _ = cs.oracle_rows(cfg, blob, scans[0], x0, abi.init_cov(1))
    c = cs.path_counts(cs.classify_rows(blob, r["ok"], r["h"], r["key"]))
    assert c[cs.HOME] == r["n_eff"] >= cs.MIN_BOX[cs.HOME] // 2 and c[cs.DESCENT] == c[cs.NEIGHBOUR] == 0
    for offset in ((0.0, 0.0, 0.0),) + cs.FAR:
        cfg, pw, pb, scans, x0 = scenes.oblique_scene(offset=offset, batch=1, n_scan=24000)
        blob = scenes.oracle_map(cfg, pw, pb)
        _, roots, nodes, _, _ = abi.parse_map_blob(blob)
        assert len(nodes) > len(roots)  # some roots were cut into octants
        r, _, _ = cs.oracle_rows(cfg, blob, scans[0], x0, abi.init_cov(1))
        c = cs.path_counts(cs.classify_rows(blob, r["ok"], r["h"], r["key"]))
        assert sum(c.values()) == r["n_eff"]
        for p, m in cs.MIN_OBLIQUE_ONE.items():  # the neighbour path too, at every offset
            assert c[p] >= m, (offset, c)
    # every oblique facet normal has all three components >= 0.2 in magnitude, none is on the grid
    for _, tilt, yaw, _, _, _ in scenes.OBLIQUE_FACETS:
        n = scenes._facet_frame(tilt, yaw)[2]
        assert np.abs(n).min() >= 0.2, n


def test_plane_tolerances_of_a_map_against_itself():
    """mapcmp.compare_blobs with per-plane tolerances 1.5 km from the origin: a map equals itself, and a normal moved by
    4x its plane's tolerance is caught."""
    cfg, pw, pb, _, _ = scenes.oblique_scene(offset=cs.FAR[0])
    blob = scenes.oracle_map(cfg, pw, pb)
    tol = cs.plane_tol_for(pw)
    st = mapcmp.compare_blobs(blob, blob, pt_atol=1e-12, var_rtol=1e-9, plane_tol=tol)
    assert st["planes"] > 500 and max(st["ratio"].values()) == 0.0
    hd, roots, nodes, aux, pts = abi.parse_map_blob(blob)
    planes = np.flatnonzero(nodes["flags"] & abi.NODE_IS_PLANE)
    tn = np.array([tol(nodes[i], aux[i], None)["normal"] for i in planes])
    i = int(planes[np.argsort(tn)[len(tn) // 2]])
    nodes = nodes.copy()
    nodes["normal"][i] += 4 * float(tn[np.argsort(tn)[len(tn) // 2]]) * np.array([1.0, -1.0, 0.0])
    with pytest.raises(AssertionError):
        mapcmp.compare_blobs(blob, abi.make_map_blob(roots, nodes, aux, pts), pt_atol=1e-12, var_rtol=1e-9, plane_tol=tol)
