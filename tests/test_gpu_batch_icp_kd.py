"""GPU: fls_match_batch for IcpOptimized and LoamPointToPlaneKdtree.

A batch runs in one cooperative launch, cut into one sub-grid and one persistent Gauss-Newton loop per scan.  Every scan of a
batch must give what its own Match gives (to fp64 rounding when the sub-grids had to be scaled down, bit for bit when the batch
fits the device) and what the CPU oracle gives.  The entries (host packed, host pcl::PointXYZI, device pointers) must agree, and the
refusals must leave the handle usable.
"""
import numpy as np
import pytest

from funny_lidar_slam_b200 import FLS_ICP_P2P, default_config, synth
from funny_lidar_slam_b200._abi import (FLS_ERR_NO_MAP, FLS_ERR_TOO_FEW_POINTS, FLS_ERR_UNSUPPORTED, FLS_FLAG_ITER_LOG, FLS_FLAG_PROFILE,
                                        FLS_LOAM_FULL, FLS_P2PLANE_KNN)
from tests.conftest import to_pcl

pytestmark = pytest.mark.gpu
FLAGS = FLS_FLAG_PROFILE | FLS_FLAG_ITER_LOG
POS_TOL, ROT_TOL = 1e-4, 1e-4
CAP = 148  # co-resident CTAs of either batch kernel that every B200 holds (ICP: 1 per SM, kd-tree: 2 per SM)
PER_CTA = {"icp": 64, "kdtree": 32}  # queries per CTA of icp_gn_kernel / loam_gn_kernel
METHOD = {"icp": FLS_ICP_P2P, "kdtree": FLS_P2PLANE_KNN}
COUNTS = ("iterations", "converged", "n_source", "n_valid")
CALL_LEVEL = ("gpu_ms", "kernel_ms", "kernel_launches", "gpu_launches", "h2d_bytes", "d2h_bytes")


def _reg(method, **kw):
    from funny_lidar_slam_b200.registration import Registration
    return Registration(default_config(method, flags=FLAGS, **kw))


def _cluster(plugin, scan):
    from funny_lidar_slam_b200.registration import PointcloudCluster
    return PointcloudCluster(ordered_cloud=scan) if plugin == "icp" else PointcloudCluster(planar_cloud=scan)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to("cuda:0")


def _log_array(g):
    return np.array([np.concatenate([d["H"].ravel(), d["g"], d["dx"], [d["sum_residual"], d["n_valid"]]]) for d in g.iter_log()])


def _single(g, plugin, scan, guess):
    T = guess.copy()
    g.Match(_cluster(plugin, scan), T)
    return T, g.last_stats, _log_array(g)


def _need(plugin, st):
    return sum(max(1, -(-x.n_source // PER_CTA[plugin])) for x in st)


def _close(a, b, tol):
    """max |a - b| <= tol, NaN only where the other one is NaN too (a scan without points has no defined pose)."""
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    d = np.abs(a - b)[~np.isnan(a)]
    return d.size == 0 or d.max() <= tol


def _check_batch_stats(st, B):
    """Call-level figures are reported on scan 0 only; algorithmic bytes on every scan that has points."""
    assert st[0].kernel_launches == 1 and st[0].gpu_launches >= 1 and st[0].gpu_ms > 0 and st[0].kernel_ms > 0
    assert st[0].h2d_bytes > 0 and st[0].d2h_bytes > 0
    for s in range(1, B):
        for f in CALL_LEVEL:
            assert getattr(st[s], f) == 0, (s, f)
    for s in range(B):
        assert (st[s].algo_bytes > 0) == (st[s].n_source > 0), s


def _features(world, pose, seed):
    from oracle import pyoracle as orc
    proj = synth.make_projected_scan(world, pose, kind="spin", sensor="vlp16", seed=seed)
    _, pi, _ = orc.extract_features(proj["depth"], proj["col"], len(proj["ordered"]), proj["row_start"], proj["row_end"], 1.0, 0.1)
    return proj["ordered"][pi].copy()


def _to_world(pts, T):
    out = pts.copy()
    out[:, :3] = (pts[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
    return out


@pytest.fixture(scope="module")
def icp_scene(world, traj, scene16):
    """Config-1 map; a ragged batch (more CTAs than the device holds) and a batch that fits."""
    v16 = {k: synth.make_scan(world, traj[k], "vlp16", seed=500 + k)["points"] for k in (3, 4, 5, 7, 8)}
    h64 = synth.make_scan(world, traj[6], "hdl64", seed=506)["points"]
    ragged = [v16[4], v16[5][::2], h64[::4], v16[7][::3], v16[3]]
    fits = [v16[5][::3], v16[4][::4], v16[8][::5]]
    return dict(map=scene16["map"], ragged=ragged, ragged_guess=np.stack([synth.perturb_pose(traj[k], seed=70 + k) for k in (4, 5, 6, 7, 3)]),
                fits=fits, fits_guess=np.stack([synth.perturb_pose(traj[k], dpos=0.1, drot_deg=1.0, seed=80 + k) for k in (5, 4, 8)]))


@pytest.fixture(scope="module")
def kd_scene(world, traj):
    """Planar-feature map of four key-frames; a ragged batch with a 0-point and a 3-point scan, and a batch that fits."""
    mp = np.concatenate([_to_world(_features(world, traj[k], k), traj[k]) for k in (3, 4, 6, 7)])
    p = {k: _features(world, traj[k], 600 + k) for k in (4, 5, 6)}
    ragged = [p[5], p[4][::2], np.zeros((0, 4), np.float32), p[6][:3].copy(), p[6][::3]]
    fits = [p[5][::15], p[4][::20], p[6][::25]]
    guess = {k: synth.perturb_pose(traj[k], dpos=0.1, drot_deg=1.0, seed=90 + k) for k in (4, 5, 6)}
    return dict(map=mp, ragged=ragged, ragged_guess=np.stack([guess[5], guess[4], guess[6], guess[6], guess[6]]),
                fits=fits, fits_guess=np.stack([guess[5], guess[4], guess[6]]))


@pytest.fixture
def scenes(icp_scene, kd_scene):
    return {"icp": icp_scene, "kdtree": kd_scene}


def _loaded(plugin, scene, **kw):
    g = _reg(METHOD[plugin], **kw)
    g.AddCloudToLocalMap([scene["map"]])
    return g


def _oracle(plugin, scene):
    from oracle import pyoracle as orc
    o = orc.Registration(default_config(METHOD[plugin]))
    o.add_cloud(scene["map"])
    return o


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_ragged_batch_matches_single_and_oracle(scenes, plugin):
    """More CTAs needed than the device holds: the sub-grids are scaled down, so sums differ from the single Match in rounding only."""
    from oracle import pyoracle as orc
    sc = scenes[plugin]
    g, o = _loaded(plugin, sc), _oracle(plugin, sc)
    scans, guesses = sc["ragged"], sc["ragged_guess"]
    conv, Tb = g.match_batch(scans, guesses)
    st = g.last_batch_stats
    _check_batch_stats(st, len(scans))
    assert _need(plugin, st) > CAP
    for s, (scan, guess) in enumerate(zip(scans, guesses)):
        T1, st1, _ = _single(g, plugin, scan, guess)
        for f in COUNTS:
            assert getattr(st[s], f) == getattr(st1, f), (s, f)
        assert bool(conv[s]) == bool(st1.converged), s
        assert _close(Tb[s], T1, 1e-9), (s, np.abs(Tb[s] - T1).max())
        if len(scan) < 50:  # the 0- and 3-point scans: nothing to compare with but their own Match
            continue
        ok_o, To, st_o = o.match(scan, guess)
        n_src = len(orc.voxel_grid(scan, g.cfg.source_cloud_filter_size)) if plugin == "icp" else len(scan)
        assert st[s].n_source == n_src, s
        assert bool(conv[s]) == ok_o and st[s].iterations == st_o.iterations and st[s].n_valid == st_o.n_valid, s
        dt, dr = synth.pose_error(Tb[s], To)
        assert dt < POS_TOL and dr < ROT_TOL, (s, dt, dr)


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_batch_that_fits_is_bitwise_single(scenes, plugin):
    """Every scan runs on the CTAs of its single Match: pose, counts and scan 0's iteration log are identical bit for bit."""
    sc = scenes[plugin]
    g = _loaded(plugin, sc)
    conv, Tb = g.match_batch(sc["fits"], sc["fits_guess"])
    st, log0 = g.last_batch_stats, _log_array(g)
    assert _need(plugin, st) <= CAP
    assert len(log0) == st[0].iterations > 0
    for s, (scan, guess) in enumerate(zip(sc["fits"], sc["fits_guess"])):
        T1, st1, log1 = _single(g, plugin, scan, guess)
        assert np.array_equal(Tb[s], T1), s
        for f in COUNTS + ("sum_residual", "algo_bytes"):
            assert getattr(st[s], f) == getattr(st1, f), (s, f)
        if s == 0:
            assert np.array_equal(log0, log1)


def test_icp_batch_of_64_scales_down(world, traj, icp_scene):
    """kMaxBatch scans, far more CTAs than the device holds: every scan still equals its single Match."""
    base = [synth.make_scan(world, traj[2 + k], "vlp16", seed=700 + k)["points"] for k in range(8)]
    scans = [base[s % 8][s % 3::1 + s % 3] for s in range(64)]
    guesses = np.stack([synth.perturb_pose(traj[2 + s % 8], dpos=0.15, drot_deg=1.5, seed=1000 + s) for s in range(64)])
    g = _loaded("icp", icp_scene)
    conv, Tb = g.match_batch(scans, guesses)
    st = g.last_batch_stats
    _check_batch_stats(st, 64)
    assert _need("icp", st) > 2 * CAP
    for s in range(64):
        T1, st1, _ = _single(g, "icp", scans[s], guesses[s])
        for f in COUNTS:
            assert getattr(st[s], f) == getattr(st1, f), (s, f)
        assert np.abs(Tb[s] - T1).max() <= 1e-9, s


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_batch_entries_agree(scenes, plugin):
    """Host packed, host pcl::PointXYZI (stride 32) and device pointers: same results, same per-scan bookkeeping."""
    sc = scenes[plugin]
    g = _loaded(plugin, sc)
    scans, guesses = sc["ragged"], sc["ragged_guess"]
    B, ns = len(scans), [len(s) for s in scans]
    d = [_dev(s) for s in scans]
    out = {"packed": g.match_batch(scans, guesses) + (g.last_batch_stats,),
           "pcl": g.match_batch([to_pcl(s) for s in scans], guesses) + (g.last_batch_stats,),
           "device": g.match_batch_device([x.data_ptr() for x in d], ns, guesses) + (g.last_batch_stats,)}
    conv0, T0, st0 = out["packed"]
    for name, (conv, Tb, st) in out.items():
        _check_batch_stats(st, B)
        assert np.array_equal(conv, conv0), name
        assert all(_close(Tb[s], T0[s], 1e-11) for s in range(B)), name
        for s in range(B):
            for f in COUNTS + ("algo_bytes",):
                assert getattr(st[s], f) == getattr(st0[s], f), (name, s, f)
        assert st[0].d2h_bytes == st0[0].d2h_bytes, name
    assert st0[0].h2d_bytes - out["device"][2][0].h2d_bytes == sum(ns) * 16
    assert out["pcl"][2][0].h2d_bytes - out["device"][2][0].h2d_bytes == sum(ns) * 32


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_batch_result_buffer(scenes, plugin):
    import torch

    from funny_lidar_slam_b200 import parallel
    sc = scenes[plugin]
    g = _loaded(plugin, sc)
    B = len(sc["ragged"])
    buf = torch.full((B * parallel.RESULT_LEN,), -7.0, dtype=torch.float64, device="cuda:0")
    g.set_result_buffer_device(buf.data_ptr(), B)
    conv, Tb = g.match_batch(sc["ragged"], sc["ragged_guess"])
    st = g.last_batch_stats
    g.set_result_buffer_device(0, 0)
    got = buf.cpu().numpy().reshape(B, parallel.RESULT_LEN)
    for s in range(B):
        Tr, ok, it = parallel.unpack_result(got[s])
        assert np.array_equal(Tr, Tb[s], equal_nan=True) and ok == bool(conv[s]) and it == st[s].iterations, s


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_fitness_after_batch_scores_scan0(scenes, plugin):
    """GetFitnessScore after a batch scores scan 0 at its final pose: as after the single Match of scan 0 (bitwise when the batch fits)."""
    sc = scenes[plugin]
    g = _loaded(plugin, sc)
    for key, exact in (("fits", True), ("ragged", False)):
        g.match_batch(sc[key], sc[key + "_guess"])
        fb = [g.GetFitnessScore(1.0), g.GetFitnessScore(2.0)]
        _single(g, plugin, sc[key][0], sc[key + "_guess"][0])
        f1 = [g.GetFitnessScore(1.0), g.GetFitnessScore(2.0)]
        assert f1[0] < 3e38 and f1[1] < 3e38, key
        for a, b in zip(fb, f1):
            assert a == b if exact else abs(a - b) <= 1e-6 * abs(b), (key, a, b)


def _status(fn):
    from funny_lidar_slam_b200._lib import FlsError
    with pytest.raises(FlsError) as e:
        fn()
    return e.value.status


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_batch_refusals(scenes, plugin):
    sc = scenes[plugin]
    scans, guesses = sc["fits"], sc["fits_guess"]
    assert _status(lambda: _reg(METHOD[plugin]).match_batch(scans, guesses)) == FLS_ERR_NO_MAP
    mapping = _loaded(plugin, sc, localization_mode=0)
    assert _status(lambda: mapping.match_batch(scans, guesses)) == FLS_ERR_UNSUPPORTED
    if plugin == "icp":  # CHECK_GT(ordered_cloud_.size(), 10u) refuses the whole call; the handle keeps matching
        g = _loaded(plugin, sc)
        conv0, T0 = g.match_batch(scans, guesses)
        assert _status(lambda: g.match_batch([scans[0], scans[1][:10], scans[2]], guesses)) == FLS_ERR_TOO_FEW_POINTS
        conv, Tb = g.match_batch(scans, guesses)
        assert np.array_equal(conv, conv0) and np.array_equal(Tb, T0)


def test_loam_full_batch_is_unsupported(kd_scene):
    g = _reg(FLS_LOAM_FULL)
    g.AddCloudToLocalMap([kd_scene["map"], kd_scene["map"][::4]])
    for B in (1, 2):
        assert _status(lambda: g.match_batch(kd_scene["fits"][:B], kd_scene["fits_guess"][:B])) == FLS_ERR_UNSUPPORTED


@pytest.mark.parametrize("plugin", ["icp", "kdtree"])
def test_batch_of_one_in_mapping_mode_is_match(world, traj, plugin):
    """A batch of one is the single Match, also in mapping mode: same poses, counts and map growth over a short stream."""
    kw = dict(localization_mode=0, local_map_size=3, dist_thre_add_cloud=0.5)
    if plugin == "icp":
        first = [synth.transform_points(synth.make_scan(world, traj[0], "vlp16", seed=60)["points"], traj[0])]
        scans = [synth.make_scan(world, traj[k], "vlp16", seed=60 + k)["points"] for k in range(1, 4)]
    else:
        first = [_to_world(_features(world, traj[k0], 100 + k0), traj[k0]) for k0 in (0, 2, 4)]
        scans = [_features(world, traj[k], 100 + k) for k in range(1, 4)]
    a, b = _reg(METHOD[plugin], **kw), _reg(METHOD[plugin], **kw)
    for c in first:
        a.AddCloudToLocalMap([c])
        b.AddCloudToLocalMap([c])
    Ta = Tb = traj[0].copy()
    for k, scan in enumerate(scans, 1):
        guess = Ta.copy() if plugin == "icp" else synth.perturb_pose(traj[k], dpos=0.05, drot_deg=0.5, seed=k)
        Ta = guess.copy()
        ok = a.Match(_cluster(plugin, scan), Ta)
        conv, Tbb = b.match_batch([scan], guess[None])
        Tb = Tbb[0]
        assert ok == bool(conv[0]) and np.array_equal(Ta, Tb), k
        for f in COUNTS + ("gpu_launches",):
            assert getattr(a.last_stats, f) == getattr(b.last_stats, f), (k, f)
        ma, mb = a.map_info(), b.map_info()
        assert (ma.n_points, ma.n_voxels, ma.bytes) == (mb.n_points, mb.n_voxels, mb.bytes), k
    assert a.map_info().n_points > 0
