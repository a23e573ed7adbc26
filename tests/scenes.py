"""Shared fixtures-as-functions for the parity tests: scenes from legkilo_b200.synth fed, unchanged,
to the CPU oracle and to the CUDA library."""
import numpy as np

import lko
from legkilo_b200 import abi, synth


def planar_scene(cfg_name="leg_fusion", n=2048, half_extent=20.0, seed_stream=2, rotvec=(2e-3, -1e-3, 3e-3),
                 trans=(0.02, -0.01, 0.03)):
    cfg = abi.CONFIGS[cfg_name]
    R, t = abi.extrinsics(cfg)
    pw, pb = synth.planar_map_points(half_extent=half_extent, ext_R=R, ext_t=t)
    o = lko.Oracle(cfg)
    o.build_voxel_map(pw, pb)
    blob = o.map_export()
    pts = synth.planar_scan(n=n, ext_R=R, ext_t=t, stream=seed_stream, rotvec=rotvec, trans=trans)
    return cfg, blob, pts


def box_scene(cfg_name="leg_fusion", lidar=None, ground_half_extent=20.0, batch=1, rot_sigma=2e-3, trans_sigma=0.02,
              streaming=False, stream0=100):
    """Box room, map built by the ORACLE's BuildVoxelMap over a small ground patch."""
    cfg, pw, pb, scans, _ = box_points(cfg_name, lidar=lidar, ground_half_extent=ground_half_extent, batch=batch,
                                       rot_sigma=rot_sigma, trans_sigma=trans_sigma, streaming=streaming, stream0=stream0)
    return cfg, oracle_map(cfg, pw, pb), scans


def box_points(cfg_name="leg_fusion", offset=None, lidar=None, ground_half_extent=20.0, batch=1, rot_sigma=2e-3,
               trans_sigma=0.02, streaming=False, stream0=100):
    """box_scene's room without the map build, optionally with its map points translated by `offset` (float32 world
    coordinates; body coordinates unchanged) and the prior there. Returns (cfg, map world f32, map body f32, scans, x0)."""
    cfg = abi.CONFIGS[cfg_name]
    R, t = abi.extrinsics(cfg)
    sc = synth.BoxScene(ground_half_extent=ground_half_extent)
    pw, pb = sc.map_points(ext_R=R, ext_t=t)
    lidar = lidar or synth.VLP16
    rv, tv = synth.random_poses(batch, rot_sigma, trans_sigma, stream=stream0)
    scans = [sc.scan(rotvec=rv[i], trans=tv[i], ext_R=R, ext_t=t, blind=cfg["blind"], stream=stream0 + 1 + i,
                     streaming=streaming, **lidar) for i in range(batch)]
    x0 = abi.default_states(batch)
    if offset is not None:
        pw = translate_f32(pw, offset)
        x0["pos"] = np.asarray(offset, np.float64)
    return cfg, pw, pb, scans, x0


def translate_f32(pw, offset):
    """World points moved by `offset` metres and stored as float32, the way the reference keeps its world cloud
    (KILO.cc:101-103): far from the origin the coordinates themselves are quantised."""
    return (np.asarray(pw, np.float64) + np.asarray(offset, np.float64)).astype(np.float32)


def _facet_frame(tilt_deg, yaw_deg):
    """Unit normal tilted `tilt_deg` from vertical towards azimuth `yaw_deg`, and two in-plane unit vectors."""
    th, ph = np.deg2rad(tilt_deg), np.deg2rad(yaw_deg)
    n = np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    u = np.cross([0.0, 0.0, 1.0], n) if tilt_deg > 1e-9 else np.array([np.cos(ph), np.sin(ph), 0.0])
    u /= np.linalg.norm(u)
    return u, np.cross(n, u), n


# (centre, tilt from vertical, azimuth, length along u, length along v, split): every normal has |component| >= 0.2,
# none is aligned to the voxel grid. The two ramps at (-1.2, -6.3) are one board 0.3 m thick: their root voxels fail
# the plane test and are cut into octants (octree descent).
#
# The last two are split-level in the map and flat in the scans: they contain the diagonal d = (1, 1, 1) resp.
# (1, -1, 1), and behind the line (p - centre) . d = 0 the map holds the facet moved SPLIT_STEP along its normal. A scan
# point there finds that moved plane in its home root voxel and is gated out by the distance (voxel_map.cc:387); the
# reference then tries one neighbour voxel (KILO.cc:156-178), which compares the voxel-unit coordinate with the voxel
# centre in metres: away from the origin that is the voxel one step along sign(p) on every axis. Where sign(p) = d
# (positive x, y, z for the first; x, z positive, y negative for the second) that neighbour lies ahead on the flat
# facet, and the row comes from it. Both sign patterns hold at the origin and, one each, 1.5 km and 12 km away.
_D111, _D1M1 = np.array([1.0, 1.0, 1.0]) / np.sqrt(3.0), np.array([1.0, -1.0, 1.0]) / np.sqrt(3.0)
SPLIT_STEP = 0.3
OBLIQUE_FACETS = (
    ((5.3, 3.1, 0.4), 35.0, 220.0, 4.0, 3.0, None),    # ramp pitched 35 deg, yawed 40 deg off the grid
    ((-4.6, 5.2, 1.1), 70.0, -65.0, 5.0, 2.5, None),   # slanted wall
    ((-5.1, -4.4, 0.2), 55.0, 25.0, 4.0, 3.5, None),   # steep ramp
    ((4.2, -5.7, 1.3), 25.0, 135.0, 4.5, 3.0, None),   # gentle ramp, leaning away
    ((-1.2, -6.3, 0.5), 40.0, 160.0, 4.0, 3.0, None),
    ((-1.2, -6.3, 0.5), 40.0, 160.0, 4.0, 3.0, "board"),  # the second face, 0.3 m along the first one's normal
    ((3.5, 6.5, 3.0), 144.7356, 45.0, 4.0, 4.0, _D111),      # n = (1, 1, -2) / sqrt(6)
    ((7.5, -3.5, 2.5), 35.2644, 63.4349, 5.0, 5.0, _D1M1),   # n = (1, 2, 1) / sqrt(6)
)


def _facet_centre(centre, tilt, yaw, split):
    return np.asarray(centre) + (0.3 * _facet_frame(tilt, yaw)[2] if isinstance(split, str) else 0.0)


def _staircase(g, origin, yaw_deg, n_steps=7, tread=0.43, riser=0.37, width=2.2, density=160.0, sigma=0.005):
    """Treads and risers of a straight staircase yawed off the grid: treads and risers share root voxels, so those
    roots fail the plane test and are cut into octants (voxel_map.cc:150-230)."""
    c, s = np.cos(np.deg2rad(yaw_deg)), np.sin(np.deg2rad(yaw_deg))
    fwd, side = np.array([c, s, 0.0]), np.array([-s, c, 0.0])
    out = []
    for k in range(n_steps):
        m = int(tread * width * density)
        a, b = g.uniform(0, tread, m), g.uniform(0, width, m)
        out.append(origin + (k * tread + a)[:, None] * fwd + b[:, None] * side +
                   np.c_[np.zeros(m), np.zeros(m), (k + 1) * riser + sigma * g.standard_normal(m)])
        m = int(riser * width * density)
        h, b = g.uniform(0, riser, m), g.uniform(0, width, m)
        out.append(origin + (k * tread + sigma * g.standard_normal(m))[:, None] * fwd + b[:, None] * side +
                   np.c_[np.zeros(m), np.zeros(m), k * riser + h])
    return np.concatenate(out)


def oblique_world_points(stream, density=160.0, sigma=0.008, stairs=True, for_map=True):
    """Points on OBLIQUE_FACETS (and a staircase yawed 27 deg) in world coordinates around the origin; for_map moves
    the split-level facets' back halves."""
    g = synth.rng(stream)
    out = []
    for centre, tilt, yaw, lu, lv, split in OBLIQUE_FACETS:
        u, v, n = _facet_frame(tilt, yaw)
        centre = _facet_centre(centre, tilt, yaw, split)
        # scans sample the split-level facets 4x as densely: few points fall where the neighbour voxel decides
        m = int(lu * lv * density * (1 if for_map or not isinstance(split, np.ndarray) else 4))
        a, b = g.uniform(-lu / 2, lu / 2, m), g.uniform(-lv / 2, lv / 2, m)
        p = centre + a[:, None] * u + b[:, None] * v + (sigma * g.standard_normal(m))[:, None] * n
        if for_map and isinstance(split, np.ndarray):
            p[(p - centre) @ split < 0] += SPLIT_STEP * n
        out.append(p)
    if stairs:
        out.append(_staircase(g, np.array([1.37, -1.83, -0.91]), 27.0, density=4 * density))
    return np.concatenate(out)


def oblique_scene(cfg_name="leg_fusion", offset=(0.0, 0.0, 0.0), batch=1, n_scan=9000, stream0=3000, rot_sigma=2e-3,
                  trans_sigma=0.02):
    """Oblique facets + staircase. Returns (cfg, map world f32 [n,3], map body f32 [n,3], scans, x0): the map is
    translated by `offset` (float32 world coordinates); scan body points are not, the prior x0 sits at `offset`."""
    cfg = abi.CONFIGS[cfg_name]
    R, t = abi.extrinsics(cfg)
    pw = oblique_world_points(stream0)
    pb32 = synth.world_to_body(pw, np.eye(3), np.zeros(3), R, t).astype(np.float32)
    pw32 = translate_f32((pb32.astype(np.float64) @ R.T) + t, offset)
    rv, tv = synth.random_poses(batch, rot_sigma, trans_sigma, stream=stream0 + 1)
    scans = []
    for i in range(batch):
        g = synth.rng(stream0 + 2 + i)
        sw = oblique_world_points(stream0 + 100 + i, density=120.0, for_map=False)
        sw = sw[g.permutation(len(sw))[:n_scan]]
        pts = np.zeros((len(sw), 4), np.float32)
        pts[:, :3] = synth.world_to_body(sw, synth.exp_so3(rv[i]), tv[i], R, t).astype(np.float32)
        scans.append(pts)
    x0 = abi.default_states(batch)
    x0["pos"] = np.asarray(offset, np.float64)
    return cfg, pw32, pb32, scans, x0


def oracle_map(cfg, pw, pb):
    """BuildVoxelMap on the CPU oracle; the exported blob."""
    o = lko.Oracle(cfg)
    o.build_voxel_map(pw, pb)
    return o.map_export()


def rel_state_err(x_a, x_b, x_prior):
    """||x_a [-] x_b||_inf / max(||x_b [-] x_prior||_inf, eps)  (SURVEY §8d pose error)."""
    num = np.abs(lko.boxminus(x_a, x_b)).max()
    den = max(np.abs(lko.boxminus(x_b, x_prior)).max(), 1e-12)
    return num / den


def rel_cov_err(P_a, P_b):
    P_a = np.asarray(P_a).reshape(30, 30)
    P_b = np.asarray(P_b).reshape(30, 30)
    return np.abs(P_a - P_b).max() / np.abs(P_b).max()
