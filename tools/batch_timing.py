#!/usr/bin/env python
"""Throughput of fls_match_batch_device for IcpOptimized and LoamPointToPlaneKdtree against the same scans as single Matches.

ICP at BASELINE config-1 shape (16-line scans vs a static map), the kd-tree point-to-plane plug-in on the planar features of
16-line scans.  For B in {1, 8, 32}: one batch call vs B single fls_match_device calls over the same device-resident scans and
guesses.  Per call: host clock around the (synchronous) call, and kernel time from FLS_FLAG_PROFILE (the GN launch only).  Every
shape is warmed up first; medians over --calls calls.  The map and the scans fit in L2 and are not flushed between calls unless
--flush-l2 (then a 256 MB buffer is overwritten before every call).  Writes one JSON file (--out) with the card name and power
limit read in the same run.

    python tools/batch_timing.py [--calls 30] [--out profiles/batch_icp_kd_n1.json] [--flush-l2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from funny_lidar_slam_b200 import _abi, synth  # noqa: E402
from funny_lidar_slam_b200.registration import Registration  # noqa: E402

SIZES = (1, 8, 32)
N_BASE = 8  # distinct scans; slot s of a batch reads scan s mod 8 with its own guess


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable: {e}"
    return dict(torch_name=name, nvidia_smi=q)


def features(world, pose, seed):
    from oracle import pyoracle as orc
    proj = synth.make_projected_scan(world, pose, kind="spin", sensor="vlp16", seed=seed)
    _, pi, _ = orc.extract_features(proj["depth"], proj["col"], len(proj["ordered"]), proj["row_start"], proj["row_end"], 1.0, 0.1)
    return proj["ordered"][pi].copy()


def to_world(pts, T):
    out = pts.copy()
    out[:, :3] = (pts[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
    return out


def scenes(world, traj):
    icp_map = synth.make_map_from_scans(world, traj[0:12:2], "vlp16", leaf=0.3)  # the scene16 map of the tests
    icp_scans = [synth.make_scan(world, traj[2 + k], "vlp16", seed=900 + k)["points"] for k in range(N_BASE)]
    kd_map = np.concatenate([to_world(features(world, traj[k], k), traj[k]) for k in (2, 4, 6, 8)])
    kd_scans = [features(world, traj[2 + k], 950 + k) for k in range(N_BASE)]
    truths = [traj[2 + k] for k in range(N_BASE)]
    return {"icp": (_abi.FLS_ICP_P2P, icp_map, icp_scans, truths), "kdtree": (_abi.FLS_P2PLANE_KNN, kd_map, kd_scans, truths)}


class Flusher:
    def __init__(self, on):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0") if on else None

    def __call__(self):
        if self.buf is not None:
            self.buf.fill_(1)
            torch.cuda.synchronize()


def measure(reg, d_scans, ns, guesses, B, calls, flush):
    """Median over `calls` of (wall us, kernel us) for one batch call and for B single calls; plus iterations of the batch."""
    ptrs = [d_scans[s % N_BASE].data_ptr() for s in range(B)]
    nb = [ns[s % N_BASE] for s in range(B)]
    G = guesses[:B]

    def batch():
        reg.match_batch_device(ptrs, nb, G)
        return reg.last_batch_stats[0].kernel_ms

    def singles():
        k = 0.0
        for s in range(B):
            reg.match_device(ptrs[s], nb[s], G[s].copy())
            k += reg.last_stats.kernel_ms
        return k

    out = {}
    for name, fn in (("batch", batch), ("singles", singles)):
        for _ in range(3):  # warm-up of this shape
            fn()
        wall, kern = [], []
        for _ in range(calls):
            flush()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            k = fn()
            wall.append((time.perf_counter() - t0) * 1e6)
            kern.append(k * 1e3)
        out[name] = dict(wall_us_median=float(np.median(wall)), wall_us_p10=float(np.percentile(wall, 10)), wall_us_p90=float(np.percentile(wall, 90)),
                         kernel_us_median=float(np.median(kern)))
    _, Tb = reg.match_batch_device(ptrs, nb, G)
    st = reg.last_batch_stats
    out["iterations"] = [int(x.iterations) for x in st]
    out["n_source"] = [int(x.n_source) for x in st]
    for name in ("batch", "singles"):
        out[name]["scans_per_s"] = B / (out[name]["wall_us_median"] * 1e-6)
    out["speedup_wall"] = out["batch"]["scans_per_s"] / out["singles"]["scans_per_s"]
    out["speedup_kernel"] = out["singles"]["kernel_us_median"] / out["batch"]["kernel_us_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "batch_icp_kd_n1.json"))
    ap.add_argument("--flush-l2", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_timing.py needs a CUDA device")
    world, traj = synth.make_world(), synth.trajectory(16)
    flush = Flusher(args.flush_l2)
    res = dict(card=card(), l2_flushed_between_calls=bool(args.flush_l2), calls_per_point=args.calls, sizes=list(SIZES),
               timing="wall = host clock around the synchronous call; kernel = FLS_FLAG_PROFILE events around the GN launch "
                      "(batch: the one launch; singles: summed over the B calls)", plugins={})
    for plugin, (method, mp, scans, truths) in scenes(world, traj).items():
        reg = Registration(_abi.default_config(method, flags=_abi.FLS_FLAG_PROFILE))
        reg.AddCloudToLocalMap([mp])
        d_scans = [torch.from_numpy(np.ascontiguousarray(s, np.float32)).to("cuda:0") for s in scans]
        ns = [len(s) for s in scans]
        guesses = np.stack([synth.perturb_pose(truths[s % N_BASE], dpos=0.1, drot_deg=1.0, seed=2000 + s) for s in range(max(SIZES))])
        res["plugins"][plugin] = dict(map_points=int(reg.map_info().n_points), scan_points=ns, by_batch={})
        for B in SIZES:
            r = measure(reg, d_scans, ns, guesses, B, args.calls, flush)
            res["plugins"][plugin]["by_batch"][str(B)] = r
            print(f"{plugin:7s} B={B:2d}: batch {r['batch']['scans_per_s']:8.0f} scans/s ({r['batch']['wall_us_median']:8.1f} us wall, "
                  f"{r['batch']['kernel_us_median']:8.1f} us kernel) | {B} singles {r['singles']['scans_per_s']:8.0f} scans/s "
                  f"({r['singles']['wall_us_median']:8.1f} us wall, {r['singles']['kernel_us_median']:8.1f} us kernel) | x{r['speedup_wall']:.2f} wall",
                  flush=True)
        reg.close()
    print(json.dumps(res["card"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
