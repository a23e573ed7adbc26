#!/usr/bin/env python
"""bench.py — LiDAR points/sec through the ESKF point-to-plane update (BASELINE.json metric).

Headline workload = BASELINE.json configs[1]: leg_fusion, 16-line Velodyne ~28.8 k pts/scan, 3 ESKF iterations,
~1.2 M-voxel map, batch = 1 per launch, one B200. One STEP = one scan through the whole hot path (3 x [residual +
all-reduce + solve] + re-projection) = ONE kernel launch. A ring of `--scans` distinct scans (default 512 = 236 MB of
points spread over 64 rooms of a 500 m x 500 m map, > the 126 MB L2) is staged in HBM; step i processes scan
i mod ring, so consecutive steps touch different points and different map regions ("inputs larger than L2").

The same JSON line also carries, inside parsed keys:
  roofline.throughput_mode  BASELINE configs[3] as this rank's shard: 128 scans x ~100 k points per launch sequence
                            against a 10 M-voxel map (the 1 024-scan batch cut 8 ways; the same 128-scan share at every N)
  e2e.stream_p50_ms         BASELINE configs[4]: p50 per-scan latency of a 10 Hz stream (~50 buckets / scan, 400 Hz
                            inertial queue, map updated after every bucket) through lk_process_scan with host buffers

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...    (one rank per GPU; scans shard, no collective on the hot path)

Prints ONE JSON line (rank 0). Point-iteration = one point through one iteration. --dump-outputs DIR writes what the
timed path returned in its last step (state, covariance, clocks, success counts, world cloud) as DIR/<name>.npy; the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
from numpy.lib import recfunctions

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "leg-kilo_b200", "python"))

from legkilo_b200 import abi, synth  # noqa: E402

ALG_BYTES_PER_POINT_ITER = 304  # SURVEY.md §8d: 16 point + 16 hash slot + 256 plane record + 16 world store

SYNTH100K = dict(n_rings=50, n_az=2048, fov_deg=(-22.5, 14.0))  # 102 400 rays, all of which hit the box

WORKLOADS = {
    # name: config, lidar, iterations, scans per launch sequence (batch), ring size, ground half extent, room grid
    "leg_fusion_b1": dict(cfg="leg_fusion", lidar="VLP16", iters=3, batch=1, ring=512, half=250.0, rooms=8,
                          baseline_config="configs[1]: leg_fusion 16-line ~28.8k pts/scan, 3 iters, ~1M-voxel map, batch=1"),
    "diter_b128": dict(cfg="diter", lidar="OS64", iters=3, batch=128, ring=128, half=250.0, rooms=8,
                       baseline_config="configs[2]: Diter++ OS-64 ~131k pts/scan, 3 iters, batch=128"),
    "synth100k_b1024": dict(cfg="leg_fusion", lidar="SYNTH100K", iters=3, batch=128, ring=128, half=250.0, rooms=8, ballast_roots=10_000_000,
                            baseline_config="configs[3]: synthetic ~100k-pt scans, 10M-voxel map, 3 iters, batch=1024 cut into "
                                            "128-scan shards (one shard per GPU; the same share at every N)"),
    "diter_b16": dict(cfg="diter", lidar="OS64", iters=3, batch=16, ring=16, half=60.0, rooms=1,
                      baseline_config="profiling-size variant of configs[2]"),
    "small": dict(cfg="leg_fusion", lidar="VLP16", iters=3, batch=1, ring=16, half=40.0, rooms=1,
                  baseline_config="smoke-size variant of configs[1]"),
}
LIDARS = dict(VLP16=synth.VLP16, OS64=synth.OS64, SYNTH100K=SYNTH100K)

DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Writes d/<name>.npy for each array: float64, point clouds float32. A cloud that would take the files past
    DUMP_BYTES is cut to a fixed, seeded sample of rows, whose indices go to d/<name>_rows.npy."""
    os.makedirs(d, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype.names:
            a = recfunctions.structured_to_unstructured(a, dtype=np.float64)
        out[name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    clouds = [k for k, a in out.items() if a.dtype == np.float32]
    room = DUMP_BYTES - sum(a.nbytes for k, a in out.items() if k not in clouds) - 256 * (len(out) + len(clouds))  # .npy headers
    for k in clouds:
        a = out[k]
        if a.nbytes <= room // len(clouds):
            continue
        keep = max(room // len(clouds), 0) // (a.nbytes // len(a) + 8)  # a row and its float64 index
        if len(a) > keep:
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            out[k] = a[rows]
            out[k + "_rows"] = rows.astype(np.float64)
    for k, a in out.items():
        np.save(os.path.join(d, k + ".npy"), a)


def ncu_traffic_family():
    """Throughput family: one iteration = pipelined kernel + fallback kernel (+ the tiny per-scan solve); their committed captures summed."""
    a, na = ncu_traffic("k_residual_stream2")
    b, _ = ncu_traffic("k_residual_fallback")
    if a is None:
        return None, None
    if b is None:
        return a, na
    return a + b, na + "; + k_residual_fallback %.3g B (the ~5 %% of the points finished in their own kernel)" % b


def ncu_traffic(kernel):
    """(dram bytes per launch, note) of the kernel's committed `ncu --set full` capture, or (None, None)."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                e = json.load(f).get(kernel)
        except (OSError, ValueError):
            e = None
        if e:
            return float(e["dram_bytes_per_launch"]), "ncu capture (%s) on: %s; algorithmic bytes of that launch %.3g" % (
                name, e["workload"], e["algorithmic_bytes_per_launch"])
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def pin_to_gpu_numa_node(local_rank):
    """Keep this rank's host threads on the CPUs local to its GPU (launch latency, page-locked copies). Returns the
    CPU list used, or None when the topology cannot be read."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        if len(bus.split(":")[0]) == 8:  # 00000000:1B:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return spec
    except Exception:  # noqa: BLE001
        return None
    return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []  # (arrival time, csv line)
        self.proc = None
        self.t_begin = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark_begin(self):
        """The timed region starts now (the sampler itself is started before the warm-up: nvidia-smi needs a few hundred
        milliseconds to come up, longer than a 20-step timed region lasts)."""
        self.t_begin = time.time()

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        t_end = time.time()
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # a sample reports the 20 ms before it arrived: keep those that overlap the timed region; when the region is
        # shorter than the sampling period and none does, the last ones before its end (the device has been under the
        # same load since the warm-up began)
        t0 = self.t_begin if self.t_begin is not None else 0.0
        rows = [r for (t, r) in self.rows if t0 <= t <= t_end + 0.06]
        window = "timed region"
        if not rows:
            rows = [r for (t, r) in self.rows if t <= t_end + 0.06][-3:]
            window = "last samples of the warm-up (timed region shorter than the 20 ms sampling period)"
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # "under load" = samples above the idle clock (the sampler also sees the gaps around the timed region)
        load = [v for v in sm if v > 500.0] or sm
        return dict(sm_mhz=float(np.median(load)) if load else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm), samples_under_load=len(load), window=window)


def build_workload(w, rank, ring):
    """Synthetic map cloud + a ring of scans. Returns dict of numpy arrays."""
    cfg = abi.CONFIGS[w["cfg"]]
    R, t = abi.extrinsics(cfg)
    rooms = synth.BoxScene.room_grid(w["rooms"]) if w["rooms"] > 1 else None
    scene = synth.BoxScene(ground_half_extent=w["half"], rooms=rooms)
    pw, pb = scene.map_points(ext_R=R, ext_t=t)
    lidar = LIDARS[w["lidar"]]
    nrooms = len(scene.rooms)
    rv, tv = synth.random_poses(ring, 2e-3 * 5, 0.02 * 5, stream=1000 + rank)  # "perturbation 5x larger" (SURVEY §8d cfg 2)
    scans = [scene.scan(rotvec=rv[i], trans=tv[i], ext_R=R, ext_t=t, blind=cfg["blind"],
                        stream=2000 + rank * 100000 + i, room=(i * 7 + rank) % nrooms, **lidar) for i in range(ring)]
    offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.uint32)
    # prior of every scan: default state placed at its room centre (the true pose is the prior perturbed by rv / tv)
    x0 = abi.default_states(ring)
    for i in range(ring):
        cx, cy = scene.rooms[(i * 7 + rank) % nrooms]
        x0["pos"][i] = (cx, cy, 0.0)
    return dict(cfg=cfg, scene=scene, map_world=pw, map_body=pb, scans=scans, pts=np.concatenate(scans),
                offs=offs, rv=rv, tv=tv, x0=x0)


def add_ballast_floors(blob, target_roots, voxel=0.5, half=250.0):
    """BASELINE configs[3] asks for a 10 M-voxel map: the rooms (built from points by BuildVoxelMap on the device) plus
    analytic plane records — extra 500 m x 500 m floors stacked 5 m apart (SURVEY §8d row 4). No scan ever sees them;
    they make the root table and the node pool as large (and as cache-unfriendly) as the config says."""
    hd, roots, nodes, aux, pts = abi.parse_map_blob(blob)
    n0 = len(roots)
    need = int(target_roots) - n0
    if need <= 0:
        return np.asarray(blob, np.uint8), n0
    # template: a ground plane record of the built map
    isp = (nodes["flags"] & 1) == 1
    cand = np.flatnonzero(isp & (np.abs(nodes["normal"][:, 2]) > 0.99))
    tpl_node = nodes[cand[len(cand) // 2]].copy()
    tpl_aux = aux[cand[len(cand) // 2]].copy()
    nv = int(round(2 * half / voxel))
    per_floor = nv * nv
    floors = (need + per_floor - 1) // per_floor
    ix, iy = np.meshgrid(np.arange(nv, dtype=np.int32), np.arange(nv, dtype=np.int32), indexing="ij")
    kx = (ix.ravel() - nv // 2).astype(np.int32)
    ky = (iy.ravel() - nv // 2).astype(np.int32)
    new_nodes, new_aux, new_roots = [], [], []
    base = len(nodes)
    made = 0
    for f in range(floors):
        m = min(per_floor, need - made)
        z_plane = -0.75 + 5.0 * (f + 2)  # above the rooms (walls end at 6.25 m)
        kz = int(np.floor(z_plane / voxel))
        nd = np.zeros(m, abi.MAP_NODE_DTYPE)
        nd[:] = tpl_node
        nd["center"][:, 0] = (kx[:m] + 0.5) * voxel
        nd["center"][:, 1] = (ky[:m] + 0.5) * voxel
        nd["center"][:, 2] = z_plane
        nd["normal"][:] = (0.0, 0.0, 1.0)
        nd["d"] = np.float32(-z_plane)
        nd["flags"] = int(tpl_node["flags"]) & 0xFF0000FB  # plane, initialised, frozen, layer 0, no children
        nd["child_base"] = -1
        ax = np.zeros(m, abi.MAP_AUX_DTYPE)
        ax[:] = tpl_aux
        ax["voxel_center"][:, 0] = (kx[:m] + 0.5) * voxel
        ax["voxel_center"][:, 1] = (ky[:m] + 0.5) * voxel
        ax["voxel_center"][:, 2] = (kz + 0.5) * voxel
        ax["pts_base"] = 0
        ax["pts_count"] = 0
        ax["new_points"] = 0
        ax["parent"] = -1
        ax["key"][:, 0] = kx[:m]; ax["key"][:, 1] = ky[:m]; ax["key"][:, 2] = kz
        rt = np.zeros(m, abi.MAP_ROOT_DTYPE)
        rt["key"] = ax["key"]
        rt["node"] = base + made + np.arange(m, dtype=np.int32)
        new_nodes.append(nd); new_aux.append(ax); new_roots.append(rt)
        made += m
    out = abi.make_map_blob(np.concatenate([roots] + new_roots), np.concatenate([nodes] + new_nodes),
                            np.concatenate([aux] + new_aux), pts)
    return out, n0 + made


def cpu_reference_run(wl, w, scan_ids, nthreads, gain_information=True):
    """The CPU restatement (oracle/) on a bounded sample: for each sampled scan the oracle builds the map of that scan's
    room from the SAME synthetic cloud (BuildVoxelMap) and runs KILO::predictUpdatePoint. Returns (seconds in the
    update loop, states, covs, n_eff, points)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lko
    cfg = wl["cfg"]
    scene = wl["scene"]
    rooms = sorted({(i * 7 + wl["rank"]) % len(scene.rooms) for i in scan_ids})
    pw, pb = wl["map_world"], wl["map_body"]
    keep = np.zeros(len(pw), bool)
    for r in rooms:
        cx, cy = scene.rooms[r]
        keep |= (np.abs(pw[:, 0] - cx) < scene.W + 2.25) & (np.abs(pw[:, 1] - cy) < scene.W + 2.25)
    cache = wl.setdefault("_oracle_cache", {})
    o = cache.get(tuple(rooms))
    if o is None:  # the map of these rooms is built once (outside every timed region) and only read afterwards
        o = lko.Oracle(cfg)
        o.build_voxel_map(pw[keep], pb[keep])
        cache[tuple(rooms)] = o
    o.set_filter(None, None, abi.process_cov_Q(cfg), None)
    n = len(scan_ids)
    pts = np.concatenate([wl["scans"][i] for i in scan_ids])
    offs = np.concatenate([[0], np.cumsum([len(wl["scans"][i]) for i in scan_ids])]).astype(np.uint32)
    sec, xo, Po, ne = o.batch_run(wl["x0"][scan_ids], abi.init_cov(n), np.zeros(n, abi.CLOCK_DTYPE), pts, offs,
                                  np.zeros(n), iters=w["iters"],
                                  gain_mode=lko.GAIN_INFORMATION if gain_information else lko.GAIN_LITERAL,
                                  nthreads=nthreads)
    return sec, xo, Po, ne, int(offs[-1])


def stream_run(cfgname, n_timed, n_warm, impl_ref, device=0, params=()):
    """BASELINE configs[4]: 10 Hz stream of scans, ~50 time buckets each, inertial (nclt: only_imu_use) or
    kinematic+inertial (leg_fusion) queue interleaved, map updated after every bucket. One STEP = one scan through
    lk_process_scan with HOST buffers (this mode is end-to-end by nature). Returns per-scan wall ms and counters."""
    from legkilo_b200 import Engine
    cfg = abi.CONFIGS[cfgname]
    R, t = abi.extrinsics(cfg)
    scene = synth.BoxScene(ground_half_extent=40.0)
    pw, pb = scene.map_points(ext_R=R, ext_t=t)
    n = n_timed + n_warm
    g = synth.rng(77)
    # a slow random walk of the true pose; the filter starts at the first true pose
    rv = np.cumsum(2e-3 * g.standard_normal((n, 3)), 0)
    tv = np.cumsum(0.01 * g.standard_normal((n, 3)), 0) * np.array([1, 1, 0.1])
    scans = [scene.scan(rotvec=rv[i], trans=tv[i], ext_R=R, ext_t=t, blind=cfg["blind"], stream=5000 + i, streaming=True,
                        **synth.VLP16) for i in range(n)]
    kin_mode = not cfg["only_imu_use"]
    Q = abi.process_cov_Q(cfg)
    if impl_ref:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import lko
        o = lko.Oracle(cfg)
        o.build_voxel_map(pw, pb)
        o.set_options(gain_mode=lko.GAIN_LITERAL, iters=1, update_map=True, imu_mode_only=not kin_mode, gravity=9.81, acc_norm=9.79)

        def proc(x, P, clk, pts, offs, times, meas, t0):
            o.set_filter(x, P, Q, clk)
            r = o.process_scan(t0, pts, imu=None if kin_mode else meas, kin=meas if kin_mode else None)
            xo, Po, _, co = o.get_filter()
            return xo, Po.reshape(1, 900), co, r["n_eff"], r["world"]
    else:
        eng = Engine(cfg, device=device)
        for kv in params:
            k, v = kv.split("=")
            eng.set_param(k, float(v))
        eng.map_build(pw, pb)

        def proc(x, P, clk, pts, offs, times, meas, t0):
            out = eng.process_scan(x, P, Q, clk, pts, offs, times, imu=None if kin_mode else meas, kin=meas if kin_mode else None,
                                   gravity=9.81, acc_norm=9.79, iters=1, update_map=True)
            return out["x"], out["P"].reshape(1, 900), out["clk"], out["n_eff"], out["world"]
    x = abi.default_states(1); P = abi.init_cov(1); clk = np.zeros(1, abi.CLOCK_DTYPE)
    lat, neff = [], []
    for i, sc in enumerate(scans):
        t0 = 0.1 * i
        pts, offs, times = synth.bucketize(sc, begin_time=t0)
        meas = (synth.kinimu_stream if kin_mode else synth.imu_stream)(t0 - 0.1 if i else -0.005, t0 + 0.1, 400.0, stream=9000 + i)
        meas = meas[meas["stamp"] > float(clk["last_update_time"][0]) - 1.0]
        a = time.perf_counter()
        x, P, clk, ne, world = proc(x, P, clk, pts, offs, times, meas, t0)
        lat.append(1e3 * (time.perf_counter() - a)); neff.append(ne)
    return dict(lat=np.array(lat[n_warm:]), neff=np.array(neff[n_warm:]), kin_mode=kin_mode,
                points_per_scan=int(np.mean([len(s) for s in scans])),
                last=dict(x=x, P=P.reshape(1, 30, 30), clk=clk, n_eff=np.array([ne]), world=world))


def stream_latency(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    cfgname = "nclt" if args.workload == "nclt_stream" else "leg_fusion"
    K, W = args.steps, max(args.warmup, 3)
    impl_ref = args.impl == "reference"
    r = stream_run(cfgname, K, W, impl_ref, device=int(os.environ.get("LOCAL_RANK", "0")), params=args.param)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["last"])
    lat = r["lat"]
    line = dict(metric="p50 per-scan latency of the streaming ESKF LiDAR update (10 Hz, ~50 buckets/scan, map updated per bucket)",
                value=float(np.median(lat)), unit="ms", n_gpus=1, steps=K, warmup=W, ms_per_step=float(np.mean(lat)),
                p95_ms=float(np.percentile(lat, 95)), higher_is_better=False, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", impl="reference" if impl_ref else "ours",
                config=dict(workload=args.workload, baseline_config="configs[4]: NCLT-style 10 Hz stream, IMU%s observations, latency mode" % ("+kinematic" if r["kin_mode"] else ""),
                            points_per_scan=r["points_per_scan"], buckets_per_scan=51, imu_hz=400, iters=1,
                            update_map=True, n_eff_mean=float(np.mean(r["neff"])),
                            note="wall clock around lk_process_scan with host buffers (H2D + D2H + sync inside)" if not impl_ref else
                                 "CPU restatement (oracle/), literal N x N gain per bucket as the reference, 1 thread"))
    print(json.dumps(line))
    return 0


def throughput_mode(args, rank, world, local_rank, dist, hbm_peak):
    """BASELINE configs[3] on this rank's shard: 128 scans x ~100 k points, 10 M-voxel map, 3 iterations; the 1 024-scan batch
    of the config is 8 such shards (no data-path collective), so the per-rank work is the same at every N (weak scaling)."""
    from legkilo_b200 import Engine
    w = WORKLOADS["synth100k_b1024"]
    B = w["batch"]
    wl = build_workload(w, rank, B)
    cfg = wl["cfg"]
    eng = Engine(cfg, device=local_rank)
    eng.map_build(wl["map_world"], wl["map_body"])
    blob, n_roots = add_ballast_floors(eng.map_download(), w["ballast_roots"], half=w["half"])
    eng.map_upload(blob)
    del blob
    mstats = eng.map_stats()
    Q = abi.process_cov_Q(cfg)
    eng.stage(wl["x0"], abi.init_cov(B), Q, np.zeros(B, abi.CLOCK_DTYPE), wl["pts"], wl["offs"], np.zeros(B))
    for _ in range(2):
        eng.run_range(0, B, iters=w["iters"])
    eng.sync()
    if dist is not None:
        dist.barrier()
    reps = 5
    eng.timer_start()
    for _ in range(reps):
        eng.run_range(0, B, iters=w["iters"])
    tb = eng.timer_stop()
    if dist is not None:
        dist.barrier()
    work = float(wl["offs"][B]) * w["iters"] * reps
    ms, total_work = tb["total_ms"], work
    if dist is not None:
        import torch
        tt = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
        ww = torch.tensor([work], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(ww, op=dist.ReduceOp.SUM)
        total_work = float(ww.item())
    rl = max(tb["residual_launches"], 1)
    rms = tb["residual_ms"] / rl
    ach = ALG_BYTES_PER_POINT_ITER * (work / rl) / (rms * 1e-3) / 1e9
    # pose check of a few scans of the shard against the CPU restatement (rank 0 only, N = 1 only)
    pose = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        wl["rank"] = rank
        ids = [0, 1]
        sec, xo, Po, ne_cpu, npts = cpu_reference_run(wl, w, ids, 1)
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import lko
        out = eng.fetch(want_world=False)
        ex = eP = 0.0
        for j, i in enumerate(ids):
            num = np.abs(lko.boxminus(out["x"][i:i + 1], xo[j:j + 1])).max()
            den = max(np.abs(lko.boxminus(xo[j:j + 1], wl["x0"][i:i + 1])).max(), 1e-12)
            ex = max(ex, num / den)
            eP = max(eP, np.abs(out["P"][i] - Po[j]).max() / np.abs(Po[j]).max())
        pose = dict(pose_rel_err_max=ex, cov_rel_err_max=eP, scans_checked=len(ids),
                    n_eff_equal=bool(np.array_equal(out["n_eff"][ids], ne_cpu)),
                    cpu_one_thread=npts * w["iters"] / sec)
    eng.close()
    return dict(workload="synth100k_b1024", baseline_config=w["baseline_config"], value=total_work / (ms * 1e-3),
                unit="point-iterations/s", frac=ach / hbm_peak, achieved=ach, peak=hbm_peak, bound="hbm",
                kernel="k_residual_stream2 + k_residual_fallback (+ k_scan_tail, the per-scan solve)", traffic=ncu_traffic_family()[0],
                ms_per_step=ms / reps, steps=reps,
                scans_per_step_per_gpu=B, points_per_scan=int(wl["offs"][B] // B), n_gpus=world, map=mstats,
                avg_launch_us=rms * 1e3, share_of_step=tb["residual_ms"] / tb["total_ms"], pose_vs_cpu=pose,
                timing="CUDA events: timed region for value (max over ranks), per-launch events for frac (this rank)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 4096, streaming workloads 100)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 512, streaming workloads 5)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="leg_fusion_b1", choices=sorted(WORKLOADS) + ["nclt_stream", "leg_fusion_stream"])
    ap.add_argument("--scans", type=int, default=0, help="ring size (distinct scans staged in HBM)")
    ap.add_argument("--e2e-steps", type=int, default=256)
    ap.add_argument("--cpu-scans", type=int, default=8)
    ap.add_argument("--stream-scans", type=int, default=40)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-throughput", action="store_true", help="skip roofline.throughput_mode (configs[3] shard)")
    ap.add_argument("--no-stream", action="store_true", help="skip e2e.stream_p50_ms (configs[4])")
    ap.add_argument("--param", action="append", default=[], help="engine parameter name=value (lk_set_param), repeatable")
    ap.add_argument("--fused", type=int, default=-1, help="0 = force the multi-kernel path for batch-of-one runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    stream = args.workload.endswith("_stream")
    if args.steps is None:
        args.steps = 100 if stream else 4096
    if args.warmup is None:
        args.warmup = 5 if stream else 512
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if stream:
        return stream_latency(args)
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ring = args.scans or w["ring"]
    ring = max(ring, w["batch"])
    K, W = args.steps, max(args.warmup, 3)
    hbm_peak, peak_src = measured_peaks()

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        ncores = os.cpu_count() or 1
        # One scan per host thread, every thread busy and pinned: the reference's per-scan loop is serial (KILO.cc:122), so
        # the only way it can use the box is independent scans side by side. One STEP = ncores scans taken room by room
        # (the oracle builds the map of those rooms only, outside the timed region).
        ring_n = min(512, max(64, 4 * ncores))
        wl = build_workload(w, 0, ring_n)
        wl["rank"] = 0
        n_rooms = len(wl["scene"].rooms)
        order = sorted(range(ring_n), key=lambda i: ((i * 7) % n_rooms, i))
        ids = order[:min(ncores, ring_n)]
        nthreads = len(ids)
        for _ in range(W):
            cpu_reference_run(wl, w, ids, nthreads)
        secs, npts = [], 0
        for _ in range(K):
            sec, xo, Po, ne, npts = cpu_reference_run(wl, w, ids, nthreads)
            secs.append(sec)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dict(x=xo, P=Po.reshape(-1, 30, 30), n_eff=ne))
        med = float(np.median(secs))
        val = npts * w["iters"] / med
        # the same loop on ONE scan with one thread: what a single scan (the step of the CUDA arm) gets from this CPU
        sec1, _, _, _, npts1 = cpu_reference_run(wl, w, ids[:2], 1)
        one_thread = npts1 * w["iters"] / sec1
        line = dict(metric="LiDAR point-iterations/sec through the ESKF point-to-plane update", value=val,
                    unit="point-iterations/s", impl="reference", n_gpus=args.gpus, steps=K, warmup=W,
                    ms_per_step=1e3 * med, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f64", data="synthetic",
                    config=dict(workload=args.workload, baseline_config=w["baseline_config"], iters=w["iters"],
                                note="CPU restatement of the reference path (oracle/, information-form gain), one scan per pinned host "
                                     "thread, %d scans side by side per step; value = work of a step / MEDIAN step time" % nthreads,
                                step_seconds=[round(s, 5) for s in secs]),
                    cpu_baseline=dict(value=val, unit="point-iterations/s", cores=nthreads, kind="port",
                                      sample=f"{len(ids)} scans x ~{len(wl['scans'][0])} pts x {w['iters']} iters per step, {K} steps (median), "
                                             f"{nthreads} pinned threads of {ncores} hardware threads",
                                      single_scan_one_thread=one_thread),
                    e2e=dict(value=val, unit="point-iterations/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (CUDA)
    numa = pin_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from legkilo_b200 import Engine, pinned_empty

    def barrier():
        if dist is not None:
            dist.barrier()

    # configs[3] shard first (throughput family): it also brings the device to its loaded clocks before the short
    # latency-mode region below
    tmode = None
    if w["batch"] == 1 and not args.no_throughput:
        tmode = throughput_mode(args, rank, world, local_rank, dist, hbm_peak)

    sampler = ClockSampler(local_rank)  # started well ahead: nvidia-smi takes a few hundred ms to deliver its first row
    sampler.start()
    t_setup = time.time()
    wl = build_workload(w, rank, ring)
    wl["rank"] = rank
    cfg = wl["cfg"]
    eng = Engine(cfg, device=local_rank)
    for kv in args.param:
        k, v = kv.split("=")
        eng.set_param(k, float(v))
    if args.fused >= 0:
        eng.set_param("fused", args.fused)
    eng.map_build(wl["map_world"], wl["map_body"])
    if w.get("ballast_roots"):
        blob, _ = add_ballast_floors(eng.map_download(), w["ballast_roots"], half=w["half"])
        eng.map_upload(blob)
        del blob
    mstats = eng.map_stats()
    nsc = ring
    Q = abi.process_cov_Q(cfg)
    x0, P0, clk0 = wl["x0"], abi.init_cov(nsc), np.zeros(nsc, abi.CLOCK_DTYPE)
    eng.stage(x0, P0, Q, clk0, wl["pts"], wl["offs"], np.zeros(nsc))
    B = w["batch"]
    groups = nsc // B  # step g processes scans [g*B, (g+1)*B)
    pts_per_group = [int(wl["offs"][(g + 1) * B] - wl["offs"][g * B]) for g in range(groups)]
    setup_s = time.time() - t_setup

    fused = (B == 1 and args.fused != 0)
    if fused:
        # one kernel per step: its average duration over the timed region is region / launches. Per-launch events
        # would sit between consecutive launches and defeat their overlap (programmatic dependent launch).
        eng.set_param("kernel_timing", 0)

    # warm-up (also warms the ring once when W >= groups)
    for i in range(W):
        eng.run_range((i % groups) * B, B, iters=w["iters"])
    eng.sync()
    barrier()
    sampler.mark_begin()
    eng.timer_start()
    work = 0
    for i in range(K):
        g = i % groups
        eng.run_range(g * B, B, iters=w["iters"])
        work += pts_per_group[g] * w["iters"]
    tm = eng.timer_stop()
    clocks = sampler.stop()
    barrier()
    if args.dump_outputs and rank == 0:
        g = (K - 1) % groups
        eng.sync()
        out = eng.fetch(want_world=True)
        o0, o1 = int(wl["offs"][g * B]), int(wl["offs"][(g + 1) * B])
        s = slice(g * B, (g + 1) * B)
        dump_outputs(args.dump_outputs, dict(x=out["x"][s], P=out["P"][s].reshape(B, 30, 30), clk=out["clk"][s],
                                             n_eff=out["n_eff"][s], world=out["world"][o0:o1]))
        del out
    elapsed_ms = tm["total_ms"]
    if dist is not None:
        import torch
        tt = torch.tensor([elapsed_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tt.item())
        ww = torch.tensor([float(work)], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(ww, op=dist.ReduceOp.SUM)
        total_work = float(ww.item())
    else:
        total_work = float(work)
    value = total_work / (elapsed_ms * 1e-3)

    # roofline of the dominant kernel: algorithmic bytes / its own event-timed duration
    r_launches = max(tm["residual_launches"], 1)
    res_total_ms = tm["total_ms"] if fused else tm["residual_ms"]
    res_ms = res_total_ms / r_launches
    alg_bytes_per_launch = ALG_BYTES_PER_POINT_ITER * (work / r_launches)
    achieved = alg_bytes_per_launch / (res_ms * 1e-3) / 1e9 if res_ms > 0 else 0.0
    traffic, traffic_note = ncu_traffic("k_scan_fused") if fused else ncu_traffic_family()
    roofline = dict(bound="hbm", kernel="k_scan_fused (whole scan: 3 x [residual + all-reduce + solve] + re-projection)" if fused else "k_residual_stream2 + k_residual_fallback (+ k_scan_tail, the per-scan solve)",
                    achieved=achieved, peak=hbm_peak, unit="GB/s", frac=achieved / hbm_peak, traffic=traffic, traffic_note=traffic_note,
                    peak_source=peak_src, alg_bytes_per_launch=alg_bytes_per_launch, avg_launch_us=res_ms * 1e3,
                    share_of_step=res_total_ms / tm["total_ms"] if tm["total_ms"] > 0 else None,
                    timing="CUDA events around the timed region / launches in it (the step is this one kernel)" if fused
                    else "CUDA events around every iteration's launches (pipelined kernel + fallback kernel + per-scan solve)",
                    throughput_mode=tmode)

    # CPU baseline (rank 0, N=1 only) on a bounded sample + pose error of the GPU against it
    cpu_baseline, pose = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ids = list(range(min(args.cpu_scans, nsc)))
        sec, xo, Po, ne_cpu, npts = cpu_reference_run(wl, w, ids, 1)
        cpu_val = npts * w["iters"] / sec
        cpu_baseline = dict(value=cpu_val, unit="point-iterations/s", cores=1, kind="port",
                            sample=f"{len(ids)} scans x ~{npts // len(ids)} pts x {w['iters']} iters, 1 thread (reference loop is serial), information-form gain",
                            host_cores_available=os.cpu_count())
        # same scans on the GPU (full map), compare state / covariance
        import lko
        if fused:
            for i in ids:
                eng.run_range(i, 1, iters=w["iters"])
        else:
            eng.run_range(0, len(ids), iters=w["iters"])
        eng.sync()
        out = eng.fetch(want_world=False)
        ex, eP = 0.0, 0.0
        for j, i in enumerate(ids):
            num = np.abs(lko.boxminus(out["x"][i:i + 1], xo[j:j + 1])).max()
            den = max(np.abs(lko.boxminus(xo[j:j + 1], x0[i:i + 1])).max(), 1e-12)
            ex = max(ex, num / den)
            eP = max(eP, np.abs(out["P"][i] - Po[j]).max() / np.abs(Po[j]).max())
        pose = dict(pose_rel_err_max=ex, cov_rel_err_max=eP, scans_checked=len(ids),
                    n_eff_equal=bool(np.array_equal(out["n_eff"][ids], ne_cpu)),
                    path="fused per-scan kernel" if fused else "batched")

    # end-to-end through the C ABI with pinned HOST buffers (H2D + D2H inside the timed region)
    e2e = None
    if (rank == 0 or world > 1) and not args.no_e2e:
        E = max(8, min(args.e2e_steps, K))
        maxp = max(pts_per_group)
        h_pts = pinned_empty((maxp, 4), np.float32)
        h_world = pinned_empty((maxp, 4), np.float32)
        Ps = abi.init_cov(B); cs = np.zeros(B, abi.CLOCK_DTYPE)
        t_e2e, work_e2e, h2d, d2h = 0.0, 0, 0, 0
        from legkilo_b200 import _p, lib
        for i in range(E + 3):
            g = i % groups
            o0, o1 = int(wl["offs"][g * B]), int(wl["offs"][(g + 1) * B])
            n = o1 - o0
            h_pts[:n] = wl["pts"][o0:o1]  # producer side (outside the timed region)
            so = (wl["offs"][g * B:(g + 1) * B + 1] - wl["offs"][g * B]).astype(np.uint32)
            sbp = np.arange(B + 1, dtype=np.uint32)
            bt = np.zeros(B)
            xi, Pi, ci = x0[g * B:(g + 1) * B].copy(), Ps.copy(), cs.copy()
            ne = np.zeros(B, np.uint32)
            # argument marshalling is the Python binding's cost, not the C ABI's: do it before the clock starts
            cargs = (eng.h, B, _p(xi), _p(Pi), _p(Q), _p(ci), _p(h_pts), _p(so), _p(sbp), _p(so), _p(bt), w["iters"], 0,
                     _p(h_world), _p(ne))
            fn = lib().lk_scan_update
            if i == 3:
                hp0 = np.zeros(8); lib().lk_debug_read(eng.h, 3, _p(hp0), 64)  # reset the host-phase counters
            t0 = time.perf_counter()
            rc = fn(*cargs)
            t1 = time.perf_counter()
            assert rc == 0, lib().lk_last_error(eng.h)
            if i >= 3:
                t_e2e += t1 - t0
                work_e2e += n * w["iters"]
                h2d = n * 16 + B * (288 + 7200 + 16) + 7200
                d2h = n * 16 + B * (288 + 7200 + 16 + 4)
        e2e_val = work_e2e / t_e2e
        if dist is not None:
            import torch
            tv = torch.tensor([e2e_val], dtype=torch.float64, device=f"cuda:{local_rank}")
            dist.all_reduce(tv, op=dist.ReduceOp.SUM)
            e2e_val = float(tv.item())
        hp = np.zeros(8); lib().lk_debug_read(eng.h, 3, _p(hp), 64)
        calls = max(hp[3], 1.0)
        e2e = dict(value=e2e_val, unit="point-iterations/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                   steps=E, us_per_step=t_e2e / E * 1e6,
                   host_phases_us=dict(stage=hp[0] / calls / 1e3, enqueue=hp[1] / calls / 1e3, wait_fetch=hp[2] / calls / 1e3),
                   note="lk_scan_update per step, pinned host buffers, wall clock incl. staging + sync")
        # configs[4]: the streaming latency mode, end to end by nature (rank 0)
        if rank == 0 and B == 1 and not args.no_stream:
            eng.close()
            sr = stream_run("nclt", max(args.stream_scans, 30), 5, False, device=local_rank, params=args.param)
            e2e["stream_p50_ms"] = float(np.median(sr["lat"]))
            e2e["stream"] = dict(workload="nclt_stream", baseline_config="configs[4]: NCLT-style 10 Hz stream, IMU observations, latency mode",
                                 scans=len(sr["lat"]), p50_ms=float(np.median(sr["lat"])), p95_ms=float(np.percentile(sr["lat"], 95)),
                                 mean_ms=float(np.mean(sr["lat"])), points_per_scan=sr["points_per_scan"], buckets_per_scan=51,
                                 imu_hz=400, iters=1, update_map=True, n_eff_mean=float(np.mean(sr["neff"])),
                                 timing="wall clock around lk_process_scan (host buffers: H2D + D2H + sync inside)")

    if rank == 0:
        line = dict(metric="LiDAR point-iterations/sec through the ESKF point-to-plane update", value=value,
                    unit="point-iterations/s", n_gpus=world, steps=K, warmup=W, ms_per_step=elapsed_ms / K,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                    config=dict(workload=args.workload, baseline_config=w["baseline_config"], iters=w["iters"],
                                scans_per_step=B, points_per_scan=int(np.mean([len(s) for s in wl["scans"]])),
                                ring_scans=nsc, ring_bytes=int(wl["pts"].nbytes), map=mstats,
                                l2_policy="inputs larger than L2: ring of distinct scans over distinct map regions",
                                parallelism=f"scans sharded over {world} GPU(s), no collective", host_cpus=numa),
                    gpu_launches=int(tm["launches"]), roofline=roofline, cpu_baseline=cpu_baseline, e2e=e2e,
                    pose_vs_cpu=pose, clocks=clocks, setup_s=setup_s)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
