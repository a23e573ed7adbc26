"""Regenerates tests/golden/ref_*.npz from the REFERENCE ITSELF: oracle/_ref/liblkref.so is the reference's own
eskf.cc / voxel_map.cc / KILO.cc compiled unmodified from /root/reference (oracle/ref/Makefile; third-party headers
stood in by oracle/ref/shim/). Run here, in the build container — the GPU box has no /root/reference and only reads the
committed fixtures (tests/test_reference_golden.py: oracle on CPU, CUDA path under -m gpu).

  ref_bucket_<cfg>.npz  one KILO::predictUpdatePoint bucket (KILO.cc:108-233) from a moving prior: the first-frame clouds
                        the map is built from, a digest of the reference's BuildVoxelMap result (mapcmp.digest: every
                        octree node, sign-canonical plane), inputs, then state / covariance / clocks / world cloud /
                        success count and the digest of the map after UpdateVoxelMap
  ref_stream_<kind>.npz one KILO::process frame (KILO.cc:356-398): ~50 buckets with the inertial (imu) or
                        kinematic-inertial (kin) queue drained in between; the cloud is stored in the order the
                        reference's own std::sort left it in
  ref_tape/<test>.npz   the reference's answers to every call tests/test_oracle_vs_reference.py makes of it
                        (tests/reftape.py), replayed where the reference library cannot be built
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in ("leg-kilo_b200/python", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))
import lkref  # noqa: E402
import mapcmp  # noqa: E402
from legkilo_b200 import abi, synth  # noqa: E402

HALF, WALL = 3.5, 2.75


def moving_state():
    x0 = abi.default_states(1)
    x0["vel"][0] = (0.4, -0.2, 0.05)
    x0["imu_w"][0] = (0.02, -0.03, 0.15)
    x0["imu_a"][0] = (0.3, 0.1, 9.7)
    x0["ba"][0] = (0.01, -0.02, 0.03)
    x0["bw"][0] = (1e-3, 2e-3, -1e-3)
    return x0


def scene(cfg_name, stream, streaming):
    cfg = abi.CONFIGS[cfg_name]
    R, t = abi.extrinsics(cfg)
    sc = synth.BoxScene(ground_half_extent=HALF, wall=WALL)
    pw, pb = sc.map_points(ext_R=R, ext_t=t)
    rv, tv = synth.random_poses(1, 2e-3, 0.02, stream=stream)
    scan = sc.scan(rotvec=rv[0], trans=tv[0], ext_R=R, ext_t=t, blind=cfg["blind"], stream=stream + 1, n_rings=16, n_az=120,
                   fov_deg=(-15.0, 15.0), streaming=streaming)
    return cfg, pw, pb, scan


def bucket(cfg_name):
    cfg, pw, pb, scan = scene(cfg_name, 9100, False)
    r = lkref.Reference(cfg, gravity=9.81, acc_norm=9.79)
    r.build_voxel_map(pw, pb)
    map0 = mapcmp.digest(r.map_export())
    x0 = moving_state(); P0 = abi.init_cov(1); Q = abi.process_cov_Q(cfg)
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 99.99; clk["last_update_time"] = 99.985
    r.set_filter(x0, P0, Q, clk)
    pts = np.ascontiguousarray(scan[:500])
    out = r.predict_update_point(100.0, pts)
    x, P, _, c = r.get_filter()
    np.savez_compressed(os.path.join(HERE, f"ref_bucket_{cfg_name}.npz"), pw=pw, pb=pb, map0=map0, x0=x0.view(np.float64), clk0=clk.view(np.float64),
                        t=100.0, pts=pts, x=x.view(np.float64), P=P, clk=c.view(np.float64), world=out["world"], n_eff=out["n_eff"],
                        map1=mapcmp.digest(r.map_export()))


def stream(kind):
    cfg, pw, pb, scan = scene("leg_fusion", 9200, True)
    r = lkref.Reference(cfg, imu_mode_only=(kind == "imu"), gravity=9.81, acc_norm=9.79)
    r.build_voxel_map(pw, pb)
    map0 = mapcmp.digest(r.map_export())
    x0 = moving_state(); P0 = abi.init_cov(1); Q = abi.process_cov_Q(cfg)
    clk = np.zeros(1, abi.CLOCK_DTYPE); clk["last_predict_time"] = 19.995; clk["last_update_time"] = 19.995
    r.set_filter(x0, P0, Q, clk)
    meas = (synth.imu_stream if kind == "imu" else synth.kinimu_stream)(19.996, 20.13)
    out = r.process(20.0, 20.1, scan, **{kind: meas})
    assert out["ok"]
    x, P, _, c = r.get_filter()
    np.savez_compressed(os.path.join(HERE, f"ref_stream_{kind}.npz"), pw=pw, pb=pb, map0=map0, x0=x0.view(np.float64), clk0=clk.view(np.float64),
                        begin=20.0, pts=out["body"], meas=meas.view(np.uint8), x=x.view(np.float64), P=P, clk=c.view(np.float64),
                        world=out["world"], n_eff=out["n_eff"], map1=mapcmp.digest(r.map_export()))


def tapes():
    import pytest
    os.environ["LKREF_TAPE"] = "record"
    assert pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_oracle_vs_reference.py")]) == 0


if __name__ == "__main__":
    bucket("leg_fusion")
    bucket("hilti")
    stream("imu")
    stream("kin")
    tapes()
    print("reference-made golden fixtures written")
