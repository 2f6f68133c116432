"""GPU: every Match entry point of a plug-in computes the same result and reports the same host bookkeeping.

The host side of Match (control tables, read-back, unpacking into T / converged / fls_match_stats, the iteration log and the
result buffer) is shared by the single-scan, batch, begin/end and device-pointer entries.  These tests pin what each entry
reports against the others.  The ICP and kd-tree plug-ins have a single entry; their per-Match figures over a short mapping
stream are stored in tests/golden/entry_consistency_streams.json, which `python -m tests.test_gpu_entry_consistency` rewrites.
"""
import json
import os

import numpy as np
import pytest

from funny_lidar_slam_b200 import FLS_ICP_P2P, FLS_NDT, FLS_P2PLANE_IVOX, default_config, synth
from funny_lidar_slam_b200._abi import FLS_FLAG_ITER_LOG, FLS_FLAG_PROFILE, FLS_LOAM_FULL, FLS_P2PLANE_KNN

pytestmark = pytest.mark.gpu
FLAGS = FLS_FLAG_PROFILE | FLS_FLAG_ITER_LOG
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "entry_consistency_streams.json")
COUNTS = ("iterations", "converged", "n_source", "n_valid", "gpu_launches", "h2d_bytes", "d2h_bytes", "kernel_launches", "algo_bytes")
CALL_LEVEL = ("gpu_ms", "kernel_ms", "kernel_launches", "gpu_launches", "h2d_bytes", "d2h_bytes")


def _reg(method, **kw):
    from funny_lidar_slam_b200.registration import Registration
    return Registration(default_config(method, flags=FLAGS, **kw))


def _cluster(**kw):
    from funny_lidar_slam_b200.registration import PointcloudCluster
    return PointcloudCluster(**kw)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to("cuda:0")


def _log_array(g):
    return np.array([np.concatenate([d["H"].ravel(), d["g"], d["dx"], [d["sum_residual"], d["n_valid"]]]) for d in g.iter_log()])


def _batch_scans(world, traj, B):
    scans = [synth.make_scan(world, traj[3 + s % 8], "vlp16", seed=300 + s)["points"][:: 1 + s % 3] for s in range(B)]
    guesses = np.stack([synth.perturb_pose(traj[3 + s % 8], seed=40 + s) for s in range(B)])
    return scans, guesses


def _check_batch_stats(st, B):
    """Call-level figures are reported on scan 0 only."""
    assert st[0].kernel_launches == 1 and st[0].gpu_launches >= 1 and st[0].gpu_ms > 0 and st[0].kernel_ms > 0
    assert st[0].h2d_bytes > 0 and st[0].d2h_bytes > 0
    for s in range(1, B):
        for f in CALL_LEVEL:
            assert getattr(st[s], f) == 0, (s, f)
    for s in range(B):
        assert st[s].algo_bytes > 0, s


def test_ivox_single_scan_entries_agree(scene16):
    """fls_match, fls_match_device and the batch entries with B = 1 run the same Match (the deterministic single-scan kernel)."""
    g = _reg(FLS_P2PLANE_IVOX)
    g.AddCloudToLocalMap([scene16["map"]])
    scan, guess = scene16["scan"], scene16["guess"]
    d = _dev(scan)
    out = {}
    T = guess.copy()
    g.Match(_cluster(planar_cloud=scan), T)
    out["match"] = (T, g.last_stats, _log_array(g))
    T = guess.copy()
    g.match_device(d.data_ptr(), len(scan), T)
    out["match_device"] = (T, g.last_stats, _log_array(g))
    _, Tb = g.match_batch([scan], guess[None])
    out["batch"] = (Tb[0], g.last_stats, _log_array(g))
    _, Tb = g.match_batch_device([d.data_ptr()], [len(scan)], guess[None])
    out["batch_device"] = (Tb[0], g.last_stats, _log_array(g))
    T0, st0, log0 = out["match"]
    assert len(log0) == st0.iterations > 0
    for name, (T, st, log) in out.items():
        assert np.array_equal(T, T0), name
        assert np.array_equal(log, log0), name
        for f in ("iterations", "converged", "n_source", "n_valid", "sum_residual", "algo_bytes", "d2h_bytes", "gpu_launches"):
            assert getattr(st, f) == getattr(st0, f), (name, f)
        assert st.kernel_launches == 1 and st.algo_bytes > 0 and st.gpu_ms > 0 and st.kernel_ms > 0, name
    for host, dev in (("match", "match_device"), ("batch", "batch_device")):
        assert out[host][1].h2d_bytes - out[dev][1].h2d_bytes == len(scan) * 16, (host, dev)


@pytest.mark.parametrize("B", [3, 8])
def test_ivox_batch_entries_agree(world, traj, scene16, B):
    import torch

    from funny_lidar_slam_b200 import parallel
    g = _reg(FLS_P2PLANE_IVOX)
    g.AddCloudToLocalMap([scene16["map"]])
    scans, guesses = _batch_scans(world, traj, B)
    d = [_dev(s) for s in scans]
    ptrs, ns = [x.data_ptr() for x in d], [len(s) for s in scans]
    buf = torch.full((B * parallel.RESULT_LEN,), -7.0, dtype=torch.float64, device="cuda:0")
    g.set_result_buffer_device(buf.data_ptr(), B)

    def begin_end():
        g.match_batch_begin(scans, guesses)
        return g.match_batch_end()

    def begin_end_device():
        g.match_batch_begin_device(ptrs, ns, guesses)
        return g.match_batch_end()

    runs = {"batch": lambda: g.match_batch(scans, guesses), "batch_device": lambda: g.match_batch_device(ptrs, ns, guesses),
            "begin_end": begin_end, "begin_end_device": begin_end_device}
    out = {}
    for name, run in runs.items():
        buf.fill_(-7.0)
        conv, Tb = run()
        st = g.last_batch_stats
        _check_batch_stats(st, B)
        got = buf.cpu().numpy().reshape(B, parallel.RESULT_LEN)
        for s in range(B):
            Tr, ok, it = parallel.unpack_result(got[s])
            assert np.array_equal(Tr, Tb[s]) and ok == bool(conv[s]) and it == st[s].iterations, (name, s)
            assert st[s].n_source == ns[s], (name, s)
        out[name] = (conv, Tb, st)
    g.set_result_buffer_device(0, 0)
    conv0, T0, st0 = out["batch"]
    for name, (conv, Tb, st) in out.items():
        assert np.array_equal(conv, conv0), name
        assert np.abs(Tb - T0).max() <= 1e-11, name
        for s in range(B):
            for f in ("iterations", "converged", "n_valid", "algo_bytes"):
                assert getattr(st[s], f) == getattr(st0[s], f), (name, s, f)
        assert st[0].d2h_bytes == st0[0].d2h_bytes, name
    for host, dev in (("batch", "batch_device"), ("begin_end", "begin_end_device")):
        assert out[host][2][0].h2d_bytes - out[dev][2][0].h2d_bytes == sum(ns) * 16, (host, dev)


def test_ndt_batch_entries_agree(world, traj, scene16):
    g = _reg(FLS_NDT)
    g.AddCloudToLocalMap([scene16["map"]])
    scan, guess = scene16["scan"], scene16["guess"]
    T = guess.copy()
    g.Match(_cluster(ordered_cloud=scan), T)
    st1, log1 = g.last_stats, _log_array(g)
    _, Tb = g.match_batch([scan], guess[None])
    assert np.array_equal(Tb[0], T) and np.array_equal(_log_array(g), log1)
    for f in COUNTS + ("sum_residual",):
        assert getattr(g.last_stats, f) == getattr(st1, f), f
    assert st1.kernel_launches == 1 and len(log1) == st1.iterations

    scans, guesses = _batch_scans(world, traj, 3)
    d = [_dev(s) for s in scans]
    conv, Tb = g.match_batch(scans, guesses)
    st = g.last_batch_stats
    conv_d, Tb_d = g.match_batch_device([x.data_ptr() for x in d], [len(s) for s in scans], guesses)
    st_d = g.last_batch_stats
    _check_batch_stats(st, 3)
    _check_batch_stats(st_d, 3)
    assert np.array_equal(conv, conv_d) and np.abs(Tb - Tb_d).max() <= 1e-11
    for s in range(3):
        for f in ("iterations", "converged", "n_source", "n_valid", "algo_bytes"):
            assert getattr(st[s], f) == getattr(st_d[s], f), (s, f)
    assert st[0].d2h_bytes == st_d[0].d2h_bytes
    assert st[0].h2d_bytes - st_d[0].h2d_bytes == sum(len(s) for s in scans) * 16


def _features(world, pose, seed):
    from oracle import pyoracle as orc
    proj = synth.make_projected_scan(world, pose, kind="spin", sensor="vlp16", seed=seed)
    ci, pi, _ = orc.extract_features(proj["depth"], proj["col"], len(proj["ordered"]), proj["row_start"], proj["row_end"], 1.0, 0.1)
    return proj["ordered"][pi].copy(), proj["ordered"][ci].copy()


def _to_world(pts, T):
    out = pts.copy()
    out[:, :3] = (pts[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
    return out


def _stream(world, traj, name):
    """Mapping-mode stream of one plug-in: after every Match its counts, pose, fitness score and map figures."""
    if name == "icp":
        g = _reg(FLS_ICP_P2P, localization_mode=0, local_map_size=3, dist_thre_add_cloud=0.5)
        g.AddCloudToLocalMap([synth.transform_points(synth.make_scan(world, traj[0], "vlp16", seed=60)["points"], traj[0])])
        clusters = [_cluster(ordered_cloud=synth.make_scan(world, traj[k], "vlp16", seed=60 + k)["points"]) for k in range(1, 6)]
        guesses = [None] * 5
    else:
        full = name == "loam_full"
        g = _reg(FLS_LOAM_FULL if full else FLS_P2PLANE_KNN, localization_mode=0, local_map_size=3, corner_local_map_size=3,
                 dist_thre_add_cloud=0.5)
        for k0 in (0, 2, 4):
            p0, c0 = _features(world, traj[k0], 100 + k0)
            g.AddCloudToLocalMap([_to_world(p0, traj[k0])] + ([_to_world(c0, traj[k0])] if full else []))
        clusters, guesses = [], []
        for k in range(1, 6):
            pk, ck = _features(world, traj[k], 100 + k)
            clusters.append(_cluster(planar_cloud=pk, corner_cloud=ck if full else None))
            guesses.append(synth.perturb_pose(traj[k], dpos=0.05, drot_deg=0.5, seed=k))
    rows, T = [], traj[0].copy()
    for c, guess in zip(clusters, guesses):
        T = T.copy() if guess is None else guess.copy()
        g.Match(c, T)
        st = g.last_stats
        mi = g.map_info()
        rows.append(dict(stats={f: int(getattr(st, f)) for f in COUNTS}, log_len=len(g.iter_log()), pose=T.ravel().tolist(),
                         fitness=g.GetFitnessScore(1.0), map=[mi.n_points, mi.n_voxels, mi.table_slots, mi.bytes]))
    return rows


STREAMS = ("icp", "kdtree", "loam_full")


@pytest.mark.parametrize("name", STREAMS)
def test_single_entry_plugin_stream_matches_golden(world, traj, name):
    with open(GOLDEN) as f:
        want = json.load(f)[name]
    got = _stream(world, traj, name)
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert a["log_len"] == a["stats"]["iterations"], k
        assert a["stats"]["kernel_launches"] == 1 and a["stats"]["algo_bytes"] > 0, k
        assert a == b, k


if __name__ == "__main__":
    import sys
    w, t = synth.make_world(), synth.trajectory(16)
    out = sys.argv[1] if len(sys.argv) > 1 else GOLDEN
    with open(out, "w") as f:
        json.dump({name: _stream(w, t, name) for name in STREAMS}, f, indent=1)
        f.write("\n")
