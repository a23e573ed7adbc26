"""Pins the CPU oracle (oracle/lko_core.cpp, a restatement) against the REFERENCE ITSELF run here: oracle/_ref/liblkref.so
is the reference's own eskf.cc / voxel_map.cc / KILO.cc compiled unmodified from /root/reference (oracle/ref/Makefile)
over stand-in third-party headers (oracle/ref/shim/: Eigen, PCL, ROS messages, glog, yaml-cpp are not in this image).

Same buffers into both; compared: calcBodyCov, init_plane, BuildVoxelMap (whole map, node by node), predictUpdatePoint
(state, covariance, clocks, world cloud, success count, map after UpdateVoxelMap), the one- and zero-residual branches,
predictUpdateImu / predictUpdateKinImu, the first frame of KILO::process (StateInitial + BuildVoxelMap) and later frames
(sort, bucket loop, queue drain). Tolerances are floating-point summation order only: the stand-in linear algebra and
the oracle's add in different orders, and eigenvector signs are free in both (mapcmp canonicalises them).

Where the library cannot be built, the reference's answers come from tests/golden/ref_tape/ (tests/reftape.py: recorded
from the same library by tests/golden/make_ref_golden.py, inputs checked against the recorded ones call by call); maps
are then compared through their summary (mapcmp.summary) instead of point by point, large world clouds on a seeded
sample of rows."""
import numpy as np
import pytest

import lko
import mapcmp
import reftape
from legkilo_b200 import abi, synth

TOL = 1e-10

lkref = None  # the reference for the running test: a reftape.Tape


@pytest.fixture(autouse=True)
def _reference(request):
    global lkref
    lkref = reftape.Tape(request.node.name)
    yield
    lkref.close()
    lkref = None


def _rel_state(xa, xb, x0):
    return np.abs(lko.boxminus(xa, xb)).max() / max(np.abs(lko.boxminus(xb, x0)).max(), 1e-12)


def _rel_cov(Pa, Pb):
    return np.abs(np.asarray(Pa) - np.asarray(Pb)).max() / np.abs(Pb).max()


def _scene(cfg_name, half=8.0, wall=6.25, stream=8200, streaming=False, n_rings=16, n_az=120):
    cfg = abi.CONFIGS[cfg_name]
    R, t = abi.extrinsics(cfg)
    sc = synth.BoxScene(ground_half_extent=half, wall=wall)
    pw, pb = sc.map_points(ext_R=R, ext_t=t)
    rv, tv = synth.random_poses(1, 2e-3, 0.02, stream=stream)
    scan = sc.scan(rotvec=rv[0], trans=tv[0], ext_R=R, ext_t=t, blind=cfg["blind"], stream=stream + 1, n_rings=n_rings,
                   n_az=n_az, fov_deg=(-15.0, 15.0), streaming=streaming)
    return cfg, pw, pb, scan


def _moving_state():
    x0 = abi.default_states(1)
    x0["vel"][0] = (0.4, -0.2, 0.05)
    x0["imu_w"][0] = (0.02, -0.03, 0.15)
    x0["imu_a"][0] = (0.3, 0.1, 9.7)
    x0["ba"][0] = (0.01, -0.02, 0.03)
    x0["bw"][0] = (1e-3, 2e-3, -1e-3)
    return x0


def _pair(cfg, pw, pb, x0, clk, imu_mode_only=True, acc_norm=9.79, **map_kw):
    o = lko.Oracle(cfg)
    r = lkref.Reference(cfg, imu_mode_only=imu_mode_only, gravity=9.81, acc_norm=acc_norm)
    o.set_options(gain_mode=lko.GAIN_LITERAL, iters=1, update_map=True, imu_mode_only=imu_mode_only, gravity=9.81, acc_norm=acc_norm)
    o.build_voxel_map(pw, pb, **map_kw)
    r.build_voxel_map(pw, pb, **map_kw)
    P0, Q = abi.init_cov(1), abi.process_cov_Q(cfg)
    for obj in (o, r):
        obj.set_filter(x0, P0, Q, clk)
    return o, r


def _same_filter(o, r, x0, tol=TOL):
    xo, Po, _, co = o.get_filter()
    xr, Pr, _, cr = r.get_filter()
    assert _rel_state(xo, xr, x0) < tol, _rel_state(xo, xr, x0)
    assert _rel_cov(Po, Pr) < tol, _rel_cov(Po, Pr)
    assert co.tobytes() == cr.tobytes()


def test_process_covariance_q_matches_init_process_cov():
    for name in ("leg_fusion", "hilti"):
        cfg = abi.CONFIGS[name]
        r = lkref.Reference(cfg)
        r.init_process_cov()  # ESKF::initProcessCovQ (eskf.cc:47-62)
        assert r.get_filter()[2].tobytes() == abi.process_cov_Q(cfg).ravel().tobytes()


def test_calc_body_cov_matches():
    g = np.random.default_rng(5)
    pts = g.uniform(-30, 30, (64, 3))
    pts[:4, 2] = 0.0  # the pb[2] == 0 -> 1e-4 patch (voxel_map.cc:23)
    for p in pts:
        co, po = lko.calc_body_cov(p, 0.02, 0.05)
        cr, pr = lkref.calc_body_cov(p, 0.02, 0.05)
        assert po.tobytes() == pr.tobytes()
        np.testing.assert_allclose(co, cr, rtol=0, atol=1e-13 * np.abs(cr).max())


@pytest.mark.parametrize("kind", ["plane", "blob", "edge"])
def test_init_plane_matches(kind):
    g = np.random.default_rng({"plane": 1, "blob": 2, "edge": 3}[kind])
    for trial in range(20):
        n = int(g.integers(6, 60))
        if kind == "plane":
            nrm = g.standard_normal(3); nrm /= np.linalg.norm(nrm)
            u = np.cross(nrm, [1.0, 0.3, -0.2]); u /= np.linalg.norm(u); v = np.cross(nrm, u)
            pw = g.uniform(-0.25, 0.25, (n, 1)) * u + g.uniform(-0.25, 0.25, (n, 1)) * v + 0.005 * g.standard_normal((n, 1)) * nrm
        elif kind == "blob":
            pw = g.uniform(-0.25, 0.25, (n, 3))
        else:  # two planes meeting: smallest eigenvalue near the threshold
            pw = g.uniform(-0.25, 0.25, (n, 3)); pw[: n // 2, 2] = 0.0; pw[n // 2:, 0] = 0.2 * g.uniform(0, 1)
        pw = pw + g.uniform(-20, 20, 3)
        A = 0.01 * g.standard_normal((n, 3, 3))
        var = A @ A.transpose(0, 2, 1) + 1e-5 * np.eye(3)
        po = lko.init_plane(pw, var.reshape(n, 9))
        pr = lkref.init_plane(pw, var.reshape(n, 9))
        assert po["is_plane"] == pr["is_plane"]
        if not pr["is_plane"]:
            continue
        s = 1.0 if np.dot(po["normal"], pr["normal"]) > 0 else -1.0
        np.testing.assert_allclose(po["center"], pr["center"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(s * po["normal"], pr["normal"], rtol=0, atol=1e-9)
        assert abs(s * po["d"] - pr["d"]) <= 2e-6 * max(1.0, abs(pr["d"]))  # d_ is a float
        assert abs(po["radius"] - pr["radius"]) <= 1e-6 * pr["radius"]
        np.testing.assert_allclose(po["eig"], pr["eig"], rtol=1e-5, atol=1e-9)
        pvo = po["plane_var"].copy(); pvo[:3, 3:] *= s; pvo[3:, :3] *= s
        assert np.abs(pvo - pr["plane_var"]).max() / np.abs(pr["plane_var"]).max() < 1e-7


@pytest.mark.parametrize("cfg_name,rot", [("leg_fusion", False), ("hilti", False), ("leg_fusion", True)])
def test_build_voxel_map_matches(cfg_name, rot):
    cfg, pw, pb, _ = _scene(cfg_name)
    kw = {}
    if rot:  # a first frame seen from a rotated pose: BuildVoxelMap's (rot * extR) term (voxel_map.cc:305-307)
        G = synth.exp_so3([0.02, -0.01, 0.7])
        R, t = abi.extrinsics(cfg)
        pw = ((pb.astype(np.float64) @ R.T + t) @ G.T + [1.5, -2.0, 0.1]).astype(np.float32)
        kw = dict(R=G, rot_cov=2e-6 * np.eye(3), pos_cov=3e-6 * np.eye(3))
    o = lko.Oracle(cfg); r = lkref.Reference(cfg)
    o.build_voxel_map(pw, pb, **kw); r.build_voxel_map(pw, pb, **kw)
    assert o.num_roots() == r.num_roots() > 100
    st = mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-7, pt_atol=0.0, var_rtol=1e-12)
    assert st["planes"] > 100 and st["points"] > 1000


@pytest.mark.parametrize("cfg_name", ["leg_fusion", "hilti"])
def test_predict_update_point_matches(cfg_name):
    """Three consecutive buckets through KILO::predictUpdatePoint (KILO.cc:108-233): predict, residuals with the
    neighbour-voxel retry, the literal n x n gain (eskf.cc:100-107), re-projection and UpdateVoxelMap."""
    cfg, pw, pb, scan = _scene(cfg_name)
    x0 = _moving_state()
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 99.99; clk["last_update_time"] = 99.985
    o, r = _pair(cfg, pw, pb, x0, clk)
    t = 100.0
    for k in range(3):
        pts = scan[k * 300:(k + 1) * 300]
        ro = o.predict_update_point(t, pts)
        rr = r.predict_update_point(t, pts)
        assert ro["n_eff"] == rr["n_eff"] > 200 and ro["updated"] == rr["updated"]
        m = reftape.kept_rows(rr["world"])
        np.testing.assert_allclose(ro["world"][m], rr["world"][m], rtol=0, atol=2e-6)  # float32 cloud: one ulp at 10 m
        assert (ro["world"][m, 3] == rr["world"][m, 3]).all()
        _same_filter(o, r, x0)
        t += 0.002
    st = mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-6, pt_atol=1e-11, var_rtol=1e-8)
    assert st["planes"] > 100


def test_single_and_zero_residual_branches_match():
    """dof_measurements == 1 takes the scalar branch (eskf.cc:92-99); no residual leaves the filter alone but still
    inserts the bucket (KILO.cc:187, :232)."""
    cfg, pw, pb, scan = _scene("leg_fusion")
    x0 = _moving_state()
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 9.99; clk["last_update_time"] = 9.99
    o, r = _pair(cfg, pw, pb, x0, clk)
    far = scan[:8].copy(); far[:, :3] += (300.0, 300.0, 50.0)  # nowhere near the map
    for pts, want in ((scan[:1], 1), (far, 0), (np.concatenate([far, scan[5:6]]), 1)):
        ro = o.predict_update_point(10.0, pts); rr = r.predict_update_point(10.0, pts)
        assert ro["n_eff"] == rr["n_eff"] == want and ro["updated"] == rr["updated"] == bool(want)
        m = reftape.kept_rows(rr["world"])
        assert (ro["world"][m, 3] == rr["world"][m, 3]).all()
        _same_filter(o, r, x0)
    mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-6, pt_atol=1e-11, var_rtol=1e-8)


@pytest.mark.parametrize("kind", ["imu", "kin"])
def test_inertial_and_kinematic_updates_match(kind):
    cfg, pw, pb, _ = _scene("leg_fusion", half=2.0)
    x0 = _moving_state()
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 3.0; clk["last_update_time"] = 2.995
    o, r = _pair(cfg, pw, pb, x0, clk, imu_mode_only=(kind == "imu"))
    meas = synth.imu_stream(3.0, 3.05) if kind == "imu" else synth.kinimu_stream(3.0, 3.05)
    for obj in (o, r):
        (obj.obs_imu if kind == "imu" else obj.obs_kinimu)(meas)
    _same_filter(o, r, x0, tol=1e-9)


def _first_frame_numpy(meas, gravity):
    """StateInitialByImu / ByKinImu::processing (state_initial.hpp:36-67, :74-105) restated with numpy."""
    acc, gyr = meas["acc"], meas["gyr"]
    mean_a, mean_w, n = acc[0].copy(), gyr[0].copy(), 1
    for a, w in zip(acc, gyr):
        mean_a += (a - mean_a) / n
        mean_w += (w - mean_w) / n
        n += 1
    acc_norm = np.linalg.norm(mean_a)
    return -mean_a / acc_norm * gravity, mean_w, acc_norm


@pytest.mark.parametrize("kind", ["imu", "kin"])
def test_process_first_frame_then_streaming_frames_match(kind):
    """KILO::process end to end (KILO.cc:316-399). Frame 0 initialises gravity / gyro bias / covariance / Q and builds
    the map from the raw cloud; frames 1-2 sort by curvature and walk the buckets, draining the inertial queue first.
    std::sort is not stable, so the oracle is fed the cloud in the order the reference's sort left it in."""
    cfg, _, pb, _ = _scene("leg_fusion", half=8.0)
    R, t = abi.extrinsics(cfg)
    sc = synth.BoxScene(ground_half_extent=8.0, wall=6.25)
    r = lkref.Reference(cfg, imu_mode_only=(kind == "imu"), gravity=9.81, initialised=False)
    mk = synth.imu_stream if kind == "imu" else synth.kinimu_stream
    raw = np.concatenate([pb, np.zeros((len(pb), 1), np.float32)], axis=1)
    m0 = mk(49.9, 50.0)
    out = r.process(49.9, 50.0, raw, **{kind: m0})
    assert out["ok"]
    grav, bw, acc_norm = _first_frame_numpy(m0, 9.81)
    assert abs(r.acc_norm() - acc_norm) < 1e-12
    xr, Pr, Qr, cr = r.get_filter()
    np.testing.assert_allclose(xr["grav"][0], grav, rtol=0, atol=1e-12)
    np.testing.assert_allclose(xr["bw"][0], bw, rtol=0, atol=1e-14)
    assert Pr.tobytes() == abi.init_cov(1).ravel().tobytes() and Qr.tobytes() == abi.process_cov_Q(cfg).ravel().tobytes()
    assert float(cr["last_predict_time"][0]) == float(cr["last_update_time"][0]) == 50.0
    # the oracle starts from the reference's own first-frame filter; its map from the same float32 world cloud
    # (KILO::pointLidarToWorld, KILO.cc:96-106: identity attitude, zero position)
    pw = (pb.astype(np.float64) @ R.T + t).astype(np.float32)
    m = reftape.kept_rows(out["world"])
    np.testing.assert_array_equal(out["world"][m, :3], pw[m])
    o = lko.Oracle(cfg)
    o.set_options(gain_mode=lko.GAIN_LITERAL, iters=1, update_map=True, imu_mode_only=(kind == "imu"), gravity=9.81, acc_norm=r.acc_norm())
    o.build_voxel_map(pw, pb, R=np.eye(3), rot_cov=Pr.reshape(30, 30)[:3, :3], pos_cov=Pr.reshape(30, 30)[3:6, 3:6])
    o.set_filter(xr, Pr, Qr, cr)
    mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-7, pt_atol=0.0, var_rtol=1e-12)
    x_init = xr.copy()
    t0 = 50.0
    for f in range(2):
        rv, tv = synth.random_poses(1, 2e-3, 0.02, stream=8300 + f)
        scan = sc.scan(rotvec=rv[0], trans=tv[0], ext_R=R, ext_t=t, blind=cfg["blind"], stream=8310 + f, n_rings=16, n_az=120,
                       fov_deg=(-15.0, 15.0), streaming=True)
        meas = mk(t0 + 0.001, t0 + 0.13, stream=60 + f)
        out = r.process(t0, t0 + 0.1, scan, **{kind: meas})
        assert out["ok"] and out["n_eff"] > 0.7 * len(scan)
        assert np.array_equal(np.sort(out["body"][:, 3]), out["body"][:, 3])  # sorted by curvature
        ro = o.process_scan(t0, out["body"], **{kind: meas})
        assert ro["n_eff"] == out["n_eff"]
        m = reftape.kept_rows(out["world"])
        np.testing.assert_allclose(ro["world"][m], out["world"][m], rtol=0, atol=2e-6)
        assert (ro["world"][m, 3] == out["world"][m, 3]).all()
        _same_filter(o, r, x_init, tol=1e-8)
        t0 += 0.1
    st = mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-5, pt_atol=1e-10, var_rtol=1e-7)
    assert st["planes"] > 100


def test_map_sliding_rule_matches():
    """VoxelMapManager::mapSliding / clearMemOutOfMap (voxel_map.cc:552-596): the numpy rule that
    tests/test_facade_compiles.py holds lk_map_slide to, checked against the reference on the same sequence."""
    cfg = dict(abi.CONFIGS["leg_fusion"], half_map_size=10, sliding_thresh=8.0)
    _, pw, pb, _ = _scene("leg_fusion")
    r = lkref.Reference(cfg)
    r.build_voxel_map(pw, pb)
    keys0 = r.root_keys()
    assert not r.map_slide([3.0, 0.0, 0.0])  # closer than sliding_thresh to the last slide position (the origin)
    assert r.num_roots() == len(keys0)
    assert r.map_slide([9.0, 1.0, 0.2])
    k = np.floor(np.array([9.0, 1.0, 0.2]) / 0.5).astype(int)
    keep = np.all((keys0 <= k + 10) & (keys0 >= k - 10), axis=1)
    assert 0 < keep.sum() < len(keys0)
    keys1 = r.root_keys()
    assert {tuple(x) for x in keys1.tolist()} == {tuple(x) for x in keys0[keep].tolist()}
    assert not r.map_slide([9.5, 1.0, 0.2])  # measured from the position of the last slide now


def _clutter(n=24000, seed=77):
    """Volumetric clutter with a thin slab and a flat sheet inside: roots fail the plane test, are cut into octants down to
    max_layer, big leaves freeze — cut_octo_tree, the freeze rules and the all-children descent of build_single_residual."""
    g = synth.rng(seed)
    pw = np.concatenate([
        g.uniform(-3, 3, (n // 2, 3)),
        np.c_[g.uniform(-3, 3, (n // 4, 2)), 0.13 + 0.002 * g.standard_normal(n // 4)],
        g.uniform(3, 5, (n // 4, 3)) * np.array([1, 1, 0.05])]).astype(np.float32)
    pb = pw.copy()
    pb[:, 2] -= 0.2
    return pw, pb


@pytest.mark.parametrize("cfg_over", [dict(), dict(voxel_size=0.4, max_layer=3, layer_init_num=(5, 4, 4, 3, 3), max_points_num=30)])
def test_cluttered_map_and_descent_residuals_match(cfg_over):
    """Octree subdivision (voxel_map.cc:139-183), frozen leaves (:125-129, :207-211) and residuals that come from the descent through
    non-plane roots with the most probable plane winning (voxel_map.cc:412-424), then UpdateVoxelMap into that subdivided map —
    also with a non-power-of-two voxel size, a deeper tree and other thresholds."""
    cfg = dict(abi.CONFIGS["leg_fusion"], **cfg_over)
    pw, pb = _clutter(n=24000 if not cfg_over else 70000)
    G = synth.exp_so3([0.01, -0.02, 0.03])
    kw = dict(R=G, rot_cov=np.diag([1e-6, 2e-6, 3e-6]), pos_cov=np.diag([4e-6, 5e-6, 6e-6]))
    x0 = _moving_state()
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 4.99; clk["last_update_time"] = 4.985
    o, r = _pair(cfg, pw, pb, x0, clk, **kw)
    st = mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-7, pt_atol=0.0, var_rtol=1e-12)
    assert st["interior"] > 50 and st["planes"] > 100
    # scan points: map points seen again with noise, from the lidar frame of the moving prior (identity attitude, zero position)
    g = synth.rng(5)
    R, t = abi.extrinsics(cfg)
    sel = g.choice(len(pw), 900, replace=False)
    body = ((pw[sel].astype(np.float64) + 0.004 * g.standard_normal((900, 3))) - t) @ R
    pts = np.c_[body, np.zeros(900)].astype(np.float32)
    tt = 5.0
    total = 0
    for k in range(3):
        ro = o.predict_update_point(tt, pts[k * 300:(k + 1) * 300]); rr = r.predict_update_point(tt, pts[k * 300:(k + 1) * 300])
        assert ro["n_eff"] == rr["n_eff"] and ro["updated"] == rr["updated"]
        total += rr["n_eff"]
        m = reftape.kept_rows(rr["world"])
        np.testing.assert_allclose(ro["world"][m], rr["world"][m], rtol=0, atol=2e-6)
        _same_filter(o, r, x0, tol=1e-9)
        tt += 0.002
    assert total > 100
    mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-6, pt_atol=1e-11, var_rtol=1e-8)


def test_leaves_fill_up_and_freeze_identically():
    """The same surface patch re-observed bucket after bucket until its leaves pass max_points_num: refit every 6th new point,
    then the freeze (`>=` on a plane leaf at voxel_map.cc:205, `>` at :234 and in init_octo_tree :125) with the retained points
    swapped away — counters, flags and planes of every node stay equal."""
    cfg, pw, pb, scan = _scene("leg_fusion", half=4.0, wall=3.25, n_az=90)
    x0 = _moving_state()
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 0.99; clk["last_update_time"] = 0.99
    o, r = _pair(cfg, pw, pb, x0, clk)
    g = synth.rng(9)
    base = scan[:160].copy()
    t = 1.0
    for k in range(14):
        pts = base.copy()
        pts[:, :3] += (0.003 * g.standard_normal((len(base), 3))).astype(np.float32)
        ro = o.predict_update_point(t, pts); rr = r.predict_update_point(t, pts)
        assert ro["n_eff"] == rr["n_eff"] > 100
        _same_filter(o, r, x0, tol=1e-8)
        t += 0.002
    bo, br = o.map_export(), r.map_export()
    st = mapcmp.compare_maps(br, bo, rtol=1e-5, pt_atol=1e-10, var_rtol=1e-7)
    nodes = mapcmp.digest(bo)  # the same structure as the reference's map (compare_maps above)
    frozen = ((nodes["flags"] & 4) == 0) & ((nodes["flags"] & 2) != 0)  # initialised, update_enable off
    assert frozen.sum() > 10 and (nodes["pts_count"][frozen] == 0).all()


from hypothesis import HealthCheck, Phase, example, given, settings  # noqa: E402
from hypothesis import strategies as st  # noqa: E402


# Which examples hypothesis generates depends on its version and on this function's source, so the tape holds the
# explicit ones: recorded and replayed alone, followed by 8 generated ones where the reference library runs.
@settings(max_examples=8, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True,
          phases=[Phase.explicit] if reftape.mode() != "live" else list(Phase))
@given(seed=st.integers(0, 10**6), kin=st.booleans(), cfg_name=st.sampled_from(["leg_fusion", "hilti", "nclt", "diter"]),
       voxel=st.sampled_from([0.5, 0.4, 0.25]), sigma=st.sampled_from([3.0, 2.0]))
@example(seed=0, kin=False, cfg_name="leg_fusion", voxel=0.5, sigma=3.0)
@example(seed=1, kin=True, cfg_name="hilti", voxel=0.4, sigma=2.0)
@example(seed=271828, kin=False, cfg_name="nclt", voxel=0.25, sigma=3.0)
@example(seed=314159, kin=True, cfg_name="diter", voxel=0.5, sigma=2.0)
@example(seed=999999, kin=False, cfg_name="hilti", voxel=0.25, sigma=2.0)
@example(seed=4242, kin=True, cfg_name="nclt", voxel=0.4, sigma=3.0)
@example(seed=77777, kin=False, cfg_name="diter", voxel=0.4, sigma=2.0)
@example(seed=123456, kin=True, cfg_name="leg_fusion", voxel=0.25, sigma=3.0)
def test_random_streaming_frames_match(seed, kin, cfg_name, voxel, sigma):
    """Randomised: dataset config (extrinsics), voxel size, gate width, observation mode, scene size, pose and sample noise — one
    KILO::process frame after BuildVoxelMap, reference vs oracle, fed in the reference's own sorted order."""
    cfg = dict(abi.CONFIGS[cfg_name], voxel_size=voxel, sigma_num=sigma)
    g = np.random.default_rng(seed)
    R, t = abi.extrinsics(cfg)
    half = float(g.uniform(3.0, 6.0))
    sc = synth.BoxScene(ground_half_extent=half, wall=half - 0.75)
    pw, pb = sc.map_points(ext_R=R, ext_t=t, stream=int(seed % 1000) + 1)
    x0 = _moving_state()
    x0["vel"][0] = g.uniform(-0.5, 0.5, 3)
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 7.995; clk["last_update_time"] = 7.995
    o, r = _pair(cfg, pw, pb, x0, clk, imu_mode_only=not kin)
    rv, tv = synth.random_poses(1, 3e-3, 0.03, stream=int(seed % 997) + 3)
    scan = sc.scan(rotvec=rv[0], trans=tv[0], ext_R=R, ext_t=t, blind=cfg["blind"], stream=int(seed % 991) + 5, n_rings=8, n_az=100,
                   fov_deg=(-15.0, 15.0), streaming=True)
    meas = (synth.kinimu_stream if kin else synth.imu_stream)(7.996, 8.13, stream=int(seed % 89) + 7)
    out = r.process(8.0, 8.1, scan, **{"kin" if kin else "imu": meas})
    assert out["ok"]
    ro = o.process_scan(8.0, out["body"], **{"kin" if kin else "imu": meas})
    assert ro["n_eff"] == out["n_eff"]
    m = reftape.kept_rows(out["world"])
    np.testing.assert_allclose(ro["world"][m], out["world"][m], rtol=0, atol=3e-6)
    _same_filter(o, r, x0, tol=1e-8)
    mapcmp.compare_maps(r.map_export(), o.map_export(), rtol=1e-5, pt_atol=1e-10, var_rtol=1e-7)


def test_state_boxminus_matches_including_small_angles():
    """State::operator- (eskf.cc:31-45) with Log (math_utils.hpp:71-76): the trace > 3 - 1e-6 and |theta| < 1e-3 branches included."""
    g = np.random.default_rng(11)
    for scale in (1.0, 1e-2, 5e-4, 1e-4, 1e-7, 0.0):
        for _ in range(6):
            a, b = abi.default_states(1), abi.default_states(1)
            Ra = synth.exp_so3(g.standard_normal(3))
            a["rot"][0] = Ra.ravel()
            b["rot"][0] = (Ra @ synth.exp_so3(scale * g.standard_normal(3))).ravel()
            for f in ("pos", "vel", "ba", "bw", "grav", "imu_a", "imu_w", "bv", "contact"):
                a[f][0] = g.standard_normal(3); b[f][0] = g.standard_normal(3)
            do, dr = lko.boxminus(b, a), lkref.boxminus(b, a)
            np.testing.assert_allclose(do, dr, rtol=0, atol=1e-15 + 1e-13 * np.abs(dr).max())
