"""Deterministic synthetic LiDAR workloads (SURVEY.md section 8d): an analytic world ray-cast exactly, shared by
the parity tests, the oracle and bench.py.  Pure numpy; nothing here touches the GPU or the oracle.

World (seed 0xC0FFEE): ground plane with +-2 cm bumps, 200 axis-aligned boxes (5-30 m footprints) and 300
vertical cylinders (r 0.1-0.5 m) spread over a 400 m x 400 m area.  Range noise N(0, 0.02 m) is drawn from a
counter-based generator keyed by (seed, frame, ray); returns closer than 1 m or farther than 100 m become exact
(0,0,0,0) rows like the invalid returns of the bundled Velodyne sweeps.  Intensity = |cos(incidence)|.
"""
import hashlib
import os
import tempfile

import numpy as np

SEED = 0xC0FFEE
SENSOR_HEIGHT = 1.8
R_MIN, R_MAX = 1.0, 100.0


def _splitmix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    z = x
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    return z ^ (z >> np.uint64(31))


def _uniform01(keys):
    return ((_splitmix64(keys) >> np.uint64(11)).astype(np.float64) + 0.5) / float(1 << 53)


def _normal(frame, n, stream=0):
    """n standard normals keyed by (SEED, frame, ray index): Box-Muller over two splitmix64 streams."""
    with np.errstate(over="ignore"):
        base = np.uint64(SEED) ^ (np.uint64(frame + 1) * np.uint64(0xD1342543DE82EF95)) ^ (np.uint64(stream) << np.uint64(56))
        idx = np.arange(n, dtype=np.uint64)
        u1 = _uniform01(base ^ (idx * np.uint64(2)))
        u2 = _uniform01(base ^ (idx * np.uint64(2) + np.uint64(1)))
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


class World:
    def __init__(self, seed=SEED, n_boxes=200, n_cyl=300, extent=200.0):
        rng = np.random.RandomState(seed & 0x7FFFFFFF)
        c = rng.uniform(-extent, extent, size=(n_boxes, 2))
        sz = rng.uniform(5.0, 30.0, size=(n_boxes, 2))
        h = rng.uniform(3.0, 20.0, size=n_boxes)
        # keep a corridor around the x axis free so the sensor never starts inside a building
        keep = np.abs(c[:, 1]) - sz[:, 1] / 2 > 4.0
        c, sz, h = c[keep], sz[keep], h[keep]
        self.box_min = np.stack([c[:, 0] - sz[:, 0] / 2, c[:, 1] - sz[:, 1] / 2, np.zeros(len(c))], 1)
        self.box_max = np.stack([c[:, 0] + sz[:, 0] / 2, c[:, 1] + sz[:, 1] / 2, h], 1)
        cc = rng.uniform(-extent, extent, size=(n_cyl, 2))
        keepc = np.abs(cc[:, 1]) > 2.5
        self.cyl_c = cc[keepc]
        self.cyl_r = rng.uniform(0.1, 0.5, size=n_cyl)[keepc]
        self.cyl_h = rng.uniform(3.0, 8.0, size=n_cyl)[keepc]

    @staticmethod
    def ground_bump(x, y):
        return 0.02 * (0.6 * np.sin(0.31 * x + 1.3) * np.cos(0.27 * y) + 0.4 * np.sin(0.73 * x - 0.41 * y + 0.5))


def beam_directions(n_beams, n_azimuth, elev_min_deg, elev_max_deg):
    el = np.radians(np.linspace(elev_min_deg, elev_max_deg, n_beams))
    az = np.linspace(0.0, 2.0 * np.pi, n_azimuth, endpoint=False)
    ce, se = np.cos(el)[:, None], np.sin(el)[:, None]
    d = np.stack([ce * np.cos(az)[None, :], ce * np.sin(az)[None, :], np.broadcast_to(se, (n_beams, n_azimuth))], -1)
    return d.reshape(-1, 3)  # ring-major: ray = beam * n_azimuth + azimuth


def pose_matrix(x, y, yaw, z=SENSOR_HEIGHT, roll=0.0, pitch=0.0):
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
    Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
    T = np.eye(4)
    T[:3, :3] = Rz @ Ry @ Rx
    T[:3, 3] = [x, y, z]
    return T


def cast_sweep(world, pose, frame, n_beams=64, n_azimuth=1875, elev=(-24.8, 2.0), noise_sigma=0.02, chunk=32768):
    """One sweep in the SENSOR frame as (n_beams*n_azimuth, 4) float32 [x, y, z, intensity]."""
    dirs_s = beam_directions(n_beams, n_azimuth, elev[0], elev[1])
    R, o = pose[:3, :3], pose[:3, 3]
    n = dirs_s.shape[0]
    t_best = np.full(n, np.inf)
    cosi = np.zeros(n)
    # cull objects that cannot be hit within R_MAX
    bc = 0.5 * (world.box_min + world.box_max)
    br = 0.5 * np.linalg.norm(world.box_max - world.box_min, axis=1)
    bsel = np.linalg.norm(bc[:, :2] - o[None, :2], axis=1) < R_MAX + br
    bmin, bmax = world.box_min[bsel], world.box_max[bsel]
    csel = np.linalg.norm(world.cyl_c - o[None, :2], axis=1) < R_MAX + 1.0
    cc, cr, ch = world.cyl_c[csel], world.cyl_r[csel], world.cyl_h[csel]
    for s in range(0, n, chunk):
        d = dirs_s[s:s + chunk] @ R.T  # world-frame directions
        m = d.shape[0]
        tb = np.full(m, np.inf)
        ci = np.zeros(m)
        # ground z = 0
        with np.errstate(divide="ignore", invalid="ignore"):
            tg = np.where(d[:, 2] < -1e-9, -o[2] / d[:, 2], np.inf)
        upd = tg < tb
        tb = np.where(upd, tg, tb)
        ci = np.where(upd, np.abs(d[:, 2]), ci)
        # boxes: slab test
        if len(bmin):
            with np.errstate(divide="ignore", invalid="ignore"):
                inv = 1.0 / d
                t0 = (bmin[None, :, :] - o[None, None, :]) * inv[:, None, :]
                t1 = (bmax[None, :, :] - o[None, None, :]) * inv[:, None, :]
            tn = np.minimum(t0, t1)
            tf = np.maximum(t0, t1)
            # reductions over the 3 slab axes written out (numpy's axis=2 reduce over a length-3 axis is very slow)
            m01 = np.maximum(tn[:, :, 0], tn[:, :, 1])
            tnear = np.maximum(m01, tn[:, :, 2])
            axis = np.where(tn[:, :, 1] > tn[:, :, 0], 1, 0)
            axis = np.where(tn[:, :, 2] > m01, 2, axis)
            tfar = np.minimum(np.minimum(tf[:, :, 0], tf[:, :, 1]), tf[:, :, 2])
            hit = (tnear <= tfar) & (tnear > 1e-6)
            tnear = np.where(hit, tnear, np.inf)
            j = np.argmin(tnear, axis=1)
            tt = tnear[np.arange(m), j]
            ax = axis[np.arange(m), j]
            upd = tt < tb
            tb = np.where(upd, tt, tb)
            ci = np.where(upd, np.abs(d[np.arange(m), ax]), ci)
        # vertical cylinders
        if len(cc):
            ox = o[0] - cc[None, :, 0]
            oy = o[1] - cc[None, :, 1]
            a = (d[:, 0] ** 2 + d[:, 1] ** 2)[:, None]
            b = 2.0 * (d[:, 0:1] * ox + d[:, 1:2] * oy)
            c = ox * ox + oy * oy - cr[None, :] ** 2
            disc = b * b - 4.0 * a * c
            with np.errstate(divide="ignore", invalid="ignore"):
                tc = (-b - np.sqrt(np.where(disc > 0, disc, np.nan))) / (2.0 * a)
            zc = o[2] + tc * d[:, 2:3]
            ok = (disc > 0) & (tc > 1e-6) & (zc >= 0.0) & (zc <= ch[None, :])
            tc = np.where(ok, tc, np.inf)
            j = np.argmin(tc, axis=1)
            tt = tc[np.arange(m), j]
            upd = tt < tb
            # incidence: normal is radial in xy
            tsafe = np.where(np.isfinite(tt), tt, 0.0)
            hx = o[0] + tsafe * d[:, 0] - cc[j, 0]
            hy = o[1] + tsafe * d[:, 1] - cc[j, 1]
            with np.errstate(divide="ignore", invalid="ignore"):
                cosc = np.abs(hx * d[:, 0] + hy * d[:, 1]) / np.maximum(np.hypot(hx, hy), 1e-9)
            tb = np.where(upd, tt, tb)
            ci = np.where(upd, np.nan_to_num(cosc), ci)
        t_best[s:s + m] = tb
        cosi[s:s + m] = ci
    rng = t_best + noise_sigma * _normal(frame, n)
    valid = np.isfinite(t_best) & (rng >= R_MIN) & (rng <= R_MAX)
    pts = dirs_s * np.where(valid, rng, 0.0)[:, None]
    # ground bumps: displace ground returns vertically by the analytic bump at the hit position
    world_xy = (pts @ R.T)[:, :2] + o[None, :2]
    is_ground = valid & (np.abs((pts @ R.T)[:, 2] + o[2]) < 0.2)
    pts[:, 2] += np.where(is_ground, World.ground_bump(world_xy[:, 0], world_xy[:, 1]), 0.0)
    out = np.zeros((n, 4), np.float32)
    out[:, :3] = np.where(valid[:, None], pts, 0.0)
    out[:, 3] = np.where(valid, cosi, 0.0)
    return out


def transform_cloud(pts, T):
    out = pts.copy()
    Tf = np.asarray(T, np.float64)
    out[:, :3] = (pts[:, :3].astype(np.float64) @ Tf[:3, :3].T + Tf[:3, 3]).astype(np.float32)
    return out


def drop_invalid(pts):
    return pts[np.any(pts[:, :3] != 0, axis=1)]


def numpy_voxel_downsample(pts, leaf):
    """Workload-generation helper only (centroid per occupied voxel, order unspecified) -- NOT a parity reference."""
    k = np.floor(pts[:, :3].astype(np.float64) / leaf).astype(np.int64)
    k -= k.min(axis=0)
    dims = k.max(axis=0) + 1
    key = (k[:, 0] * dims[1] + k[:, 1]) * dims[2] + k[:, 2]
    uniq, inv = np.unique(key, return_inverse=True)
    cnt = np.bincount(inv).astype(np.float64)
    out = np.empty((len(uniq), 4), np.float32)
    for c in range(4):
        out[:, c] = (np.bincount(inv, weights=pts[:, c].astype(np.float64)) / cnt).astype(np.float32)
    return out


def trajectory_pose(k, spacing=1.0):
    """Keyframe k of the synthetic drive: along +x with a gentle weave."""
    x = k * spacing
    return pose_matrix(x, 0.8 * np.sin(0.05 * x), 0.03 * np.sin(0.07 * x))


def _cache_dir():
    # one directory per user: the temporary directory is shared, and a cache another account created there is not writable
    d = os.environ.get("LGS_SYNTH_CACHE") or os.path.join(tempfile.gettempdir(), "lgs_synth_cache_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    return d


def _cached(name, params, fn):
    tag = hashlib.sha1(repr((name, params)).encode()).hexdigest()[:16]
    path = os.path.join(_cache_dir(), "%s_%s.npz" % (name, tag))
    if os.path.exists(path):
        try:
            z = np.load(path)
            return {k: z[k] for k in z.files}
        except Exception:
            pass
    out = fn()
    tmp = path + ".tmp%d.npz" % os.getpid()
    try:
        np.savez(tmp, **out)
        os.replace(tmp, path)
    except OSError:  # the cache only saves time: a full or read-only disk must not fail the run
        pass
    return out


def ndt_scan_to_map(n_map=1_000_000, n_keyframes=20, n_beams=64, n_azimuth=1875, map_leaf=0.2, seed=SEED, perturb_seed=1):
    """cfg 0: one 64-beam sweep (120 000 rays, sensor frame) against a local map of `n_keyframes` previous keyframe
    sweeps (1 m spacing, each voxel-filtered at `map_leaf`), resampled to exactly `n_map` points.
    Returns dict(source, target, T_true (map <- sensor), guess)."""

    def make():
        w = World(seed)
        clouds = []
        k = 0
        total = 0
        while k < n_keyframes or total < n_map:
            pose = trajectory_pose(k)
            sw = drop_invalid(cast_sweep(w, pose, frame=k, n_beams=n_beams, n_azimuth=n_azimuth))
            ds = numpy_voxel_downsample(sw, map_leaf)
            clouds.append(transform_cloud(ds, pose))
            total += len(ds)
            k += 1
            if k > 4 * n_keyframes + 64:
                break
        target = np.concatenate(clouds, 0)
        if len(target) > n_map:
            sel = np.sort(np.random.RandomState(seed & 0xFFFF).permutation(len(target))[:n_map])
            target = target[sel]
        pose_s = trajectory_pose(k - 1 + 0.5)
        source = cast_sweep(w, pose_s, frame=10_000, n_beams=n_beams, n_azimuth=n_azimuth)
        rs = np.random.RandomState(perturb_seed)
        d = np.array([0.3, 0.3, 0.05, np.radians(0.5), np.radians(0.5), np.radians(2.0)]) * rs.uniform(-1, 1, 6)
        P = pose_matrix(d[0], d[1], d[5], z=d[2], roll=d[3], pitch=d[4])
        guess = pose_s @ P
        return dict(source=source, target=np.ascontiguousarray(target, np.float32), T_true=pose_s, guess=guess.astype(np.float32),
                    n_keyframes_used=np.int64(k))

    return _cached("ndt_scan_to_map", (n_map, n_keyframes, n_beams, n_azimuth, map_leaf, seed, perturb_seed, 4), make)


def ndt_sweep_pool(d, n_sweeps, n_beams=64, n_azimuth=1875, seed=SEED, perturb_seed=1):
    """Further scans of the cfg 0 sequence against the same local map `d` (an ndt_scan_to_map result): sweeps re-cast
    from poses 0.5 m apart behind the first one, each with its own range noise and its own perturbed guess.
    Returns (sweeps, guesses, true_poses) including d's own sweep first."""
    w = World(seed)
    k = int(d["n_keyframes_used"])
    sweeps, guesses, poses = [d["source"]], [d["guess"]], [d["T_true"]]
    rs = np.random.RandomState(1000 + perturb_seed)
    for j in range(1, n_sweeps):
        pose = trajectory_pose(k - 1 + 0.5 - 0.5 * j)
        sweeps.append(cast_sweep(w, pose, frame=10_000 + j, n_beams=n_beams, n_azimuth=n_azimuth))
        dd = np.array([0.3, 0.3, 0.05, np.radians(0.5), np.radians(0.5), np.radians(2.0)]) * rs.uniform(-1, 1, 6)
        P = pose_matrix(dd[0], dd[1], dd[5], z=dd[2], roll=dd[3], pitch=dd[4])
        guesses.append((pose @ P).astype(np.float32))
        poses.append(pose)
    return sweeps, guesses, poses


def prefilter_sweeps(n_sweeps=4, n_beams=128, n_azimuth=2048, seed=SEED):
    """cfg 1: 128-beam sweeps of 262 144 rays (invalid returns kept as zero rows, as a driver would publish them)."""

    def make():
        w = World(seed)
        return {"sweep%d" % k: cast_sweep(w, trajectory_pose(3 * k), frame=20_000 + k, n_beams=n_beams, n_azimuth=n_azimuth, elev=(-25.0, 15.0))
                for k in range(n_sweeps)}

    d = _cached("prefilter_sweeps", (n_sweeps, n_beams, n_azimuth, seed, 3), make)
    return [d["sweep%d" % k] for k in range(n_sweeps)]


def odometry_sequence(n_sweeps=8, n_beams=64, n_azimuth=1875, spacing=1.0, seed=SEED):
    """cfg 2: consecutive sweeps along the drive with their true poses (sensor -> world)."""

    def make():
        w = World(seed)
        out = {}
        for k in range(n_sweeps):
            pose = trajectory_pose(k, spacing)
            out["sweep%d" % k] = cast_sweep(w, pose, frame=30_000 + k, n_beams=n_beams, n_azimuth=n_azimuth)
            out["pose%d" % k] = pose
        return out

    d = _cached("odometry_sequence", (n_sweeps, n_beams, n_azimuth, spacing, seed, 3), make)
    return [d["sweep%d" % k] for k in range(n_sweeps)], [d["pose%d" % k] for k in range(n_sweeps)]


# ---- cfg 2 at its full size: 1000 sweeps along a 1 km drive ------------------------------------------------------------------
LONG_WORLD = dict(n_boxes=1800, n_cyl=2700, extent=600.0)  # the 400 m world's density over 1200 m x 1200 m


def long_drive_pose(k, n_sweeps=1000, spacing=1.0):
    """Pose of sweep k of the long drive: the 1 km spline of SURVEY section 8d, centred in the large world."""
    x = (k - n_sweeps / 2) * spacing
    return pose_matrix(x, 0.8 * np.sin(0.05 * x), 0.03 * np.sin(0.07 * x))


def cast_sweep_torch(world, pose, frame, device, n_beams=64, n_azimuth=1875, elev=(-24.8, 2.0), noise_sigma=0.02):
    """cast_sweep with the ray / primitive tests as torch ops on `device` (the same geometry, f64; the range noise is the
    same counter-based stream, drawn with numpy).  Thousand-sweep workloads (cfg 2) are cast in seconds instead of tens of
    minutes.  Test-data generation only: the product never calls this.  Returns a float32 (n, 4) tensor on `device`."""
    import torch
    f64 = torch.float64
    dirs_s = torch.from_numpy(beam_directions(n_beams, n_azimuth, elev[0], elev[1])).to(device)
    R = torch.from_numpy(np.ascontiguousarray(pose[:3, :3])).to(device)
    o_np = pose[:3, 3]
    n = dirs_s.shape[0]
    bc = 0.5 * (world.box_min + world.box_max)
    br = 0.5 * np.linalg.norm(world.box_max - world.box_min, axis=1)
    bsel = np.linalg.norm(bc[:, :2] - o_np[None, :2], axis=1) < R_MAX + br
    csel = np.linalg.norm(world.cyl_c - o_np[None, :2], axis=1) < R_MAX + 1.0
    bmin = torch.from_numpy(world.box_min[bsel]).to(device)
    bmax = torch.from_numpy(world.box_max[bsel]).to(device)
    cc = torch.from_numpy(world.cyl_c[csel]).to(device)
    cr = torch.from_numpy(world.cyl_r[csel]).to(device)
    ch = torch.from_numpy(world.cyl_h[csel]).to(device)
    o = torch.from_numpy(np.ascontiguousarray(o_np)).to(device)
    inf = torch.tensor(float("inf"), dtype=f64, device=device)
    d = dirs_s @ R.T
    tg = torch.where(d[:, 2] < -1e-9, -o[2] / d[:, 2], inf)
    tb = tg.clone()
    ci = torch.where(torch.isfinite(tg), d[:, 2].abs(), torch.zeros_like(tg))
    ar = torch.arange(n, device=device)
    if bmin.shape[0]:
        inv = 1.0 / d
        t0 = (bmin[None, :, :] - o[None, None, :]) * inv[:, None, :]
        t1 = (bmax[None, :, :] - o[None, None, :]) * inv[:, None, :]
        tn, tf = torch.minimum(t0, t1), torch.maximum(t0, t1)
        m01 = torch.maximum(tn[:, :, 0], tn[:, :, 1])
        tnear = torch.maximum(m01, tn[:, :, 2])
        axis = torch.where(tn[:, :, 1] > tn[:, :, 0], 1, 0)
        axis = torch.where(tn[:, :, 2] > m01, 2, axis)
        tfar = torch.minimum(torch.minimum(tf[:, :, 0], tf[:, :, 1]), tf[:, :, 2])
        hit = (tnear <= tfar) & (tnear > 1e-6)
        tnear = torch.where(hit, tnear, inf)
        tt, j = tnear.min(dim=1)
        ax = axis[ar, j]
        upd = tt < tb
        tb = torch.where(upd, tt, tb)
        ci = torch.where(upd, d[ar, ax].abs(), ci)
    if cc.shape[0]:
        ox, oy = o[0] - cc[None, :, 0], o[1] - cc[None, :, 1]
        a = (d[:, 0] ** 2 + d[:, 1] ** 2)[:, None]
        b = 2.0 * (d[:, 0:1] * ox + d[:, 1:2] * oy)
        c = ox * ox + oy * oy - cr[None, :] ** 2
        disc = b * b - 4.0 * a * c
        tc = (-b - torch.sqrt(torch.where(disc > 0, disc, torch.full_like(disc, float("nan"))))) / (2.0 * a)
        zc = o[2] + tc * d[:, 2:3]
        ok = (disc > 0) & (tc > 1e-6) & (zc >= 0.0) & (zc <= ch[None, :])
        tc = torch.where(ok, tc, inf)
        tt, j = tc.min(dim=1)
        upd = tt < tb
        tsafe = torch.where(torch.isfinite(tt), tt, torch.zeros_like(tt))
        hx = o[0] + tsafe * d[:, 0] - cc[j, 0]
        hy = o[1] + tsafe * d[:, 1] - cc[j, 1]
        cosc = (hx * d[:, 0] + hy * d[:, 1]).abs() / torch.clamp(torch.hypot(hx, hy), min=1e-9)
        tb = torch.where(upd, tt, tb)
        ci = torch.where(upd, torch.nan_to_num(cosc), ci)
    rng = tb + noise_sigma * torch.from_numpy(_normal(frame, n)).to(device)
    valid = torch.isfinite(tb) & (rng >= R_MIN) & (rng <= R_MAX)
    pts = dirs_s * torch.where(valid, rng, torch.zeros_like(rng))[:, None]
    pw = pts @ R.T
    wx, wy = pw[:, 0] + o[0], pw[:, 1] + o[1]
    is_ground = valid & ((pw[:, 2] + o[2]).abs() < 0.2)
    bump = 0.02 * (0.6 * torch.sin(0.31 * wx + 1.3) * torch.cos(0.27 * wy) + 0.4 * torch.sin(0.73 * wx - 0.41 * wy + 0.5))
    pts[:, 2] += torch.where(is_ground, bump, torch.zeros_like(bump))
    out = torch.zeros((n, 4), dtype=torch.float32, device=device)
    out[:, :3] = torch.where(valid[:, None], pts, torch.zeros_like(pts)).to(torch.float32)
    out[:, 3] = torch.where(valid, ci, torch.zeros_like(ci)).to(torch.float32)
    return out


def long_drive(n_sweeps=1000, device="cuda", n_beams=64, n_azimuth=1875, spacing=1.0, seed=SEED):
    """cfg 2: `n_sweeps` consecutive 64-beam sweeps (120 000 rays each) 1 m apart along the 1 km spline, with their true
    poses.  Returns (float32 tensor (n_sweeps, n_rays, 4) on `device`, list of 4x4 poses)."""
    import torch
    w = World(seed, **LONG_WORLD)
    poses = [long_drive_pose(k, n_sweeps, spacing) for k in range(n_sweeps)]
    out = torch.empty((n_sweeps, n_beams * n_azimuth, 4), dtype=torch.float32, device=device)
    for k in range(n_sweeps):
        out[k] = cast_sweep_torch(w, poses[k], 60_000 + k, device, n_beams=n_beams, n_azimuth=n_azimuth)
    return out, poses


def loop_pairs(n_pairs=8, n_keyframes=41, n_beams=64, n_azimuth=1875, scan_leaf=0.2, key_leaf=0.2, seed=SEED, n_unique=4):
    """cfg 4: (scan, submap) candidate pairs.  scan = scan_leaf-filtered sweep expressed in the map frame with a
    seeded offset <= (2 m, 5 deg) from its true pose; submap = concatenation of `n_keyframes` consecutive keyframe
    clouds (each key_leaf-filtered) in the map frame, NOT yet voxel-filtered at 0.5 m (the batch API does that,
    GBS:311-313).  `n_unique` distinct places are generated and cycled with fresh offsets to reach `n_pairs`.
    Returns (scans, submaps, true_corrections) where true_correction maps the offset scan back onto the map."""

    def make():
        w = World(seed)
        out = {}
        for u in range(n_unique):
            base = 30 * u
            clouds = []
            for k in range(n_keyframes):
                pose = trajectory_pose(base + k)
                sw = drop_invalid(cast_sweep(w, pose, frame=40_000 + base + k, n_beams=n_beams, n_azimuth=n_azimuth))
                clouds.append(transform_cloud(numpy_voxel_downsample(sw, key_leaf), pose))
            out["submap%d" % u] = np.concatenate(clouds, 0)
            pose_s = trajectory_pose(base + n_keyframes // 2 + 0.4)
            sw = drop_invalid(cast_sweep(w, pose_s, frame=50_000 + u, n_beams=n_beams, n_azimuth=n_azimuth))
            out["scan%d" % u] = numpy_voxel_downsample(sw, scan_leaf)
            out["pose%d" % u] = pose_s
        return out

    d = _cached("loop_pairs", (n_keyframes, n_beams, n_azimuth, scan_leaf, key_leaf, seed, n_unique, 3), make)
    scans, submaps, corrections = [], [], []
    for i in range(n_pairs):
        u = i % n_unique
        rs = np.random.RandomState(1000 + i)
        dxy = rs.uniform(-1, 1, 2) * 2.0 / np.sqrt(2)
        yaw = np.radians(5.0) * rs.uniform(-1, 1)
        off = pose_matrix(dxy[0], dxy[1], yaw, z=0.0)
        pose_bad = off @ d["pose%d" % u]
        scans.append(transform_cloud(d["scan%d" % u], pose_bad))
        submaps.append(d["submap%d" % u])
        corrections.append(np.linalg.inv(off))
    return scans, submaps, corrections


def loop_keyframes(n_pairs=8, n_keyframes=41, n_beams=64, n_azimuth=1875, scan_leaf=0.2, key_leaf=0.2, seed=SEED, n_unique=4):
    """cfg 4 in key-frame form (what graph_based_slam holds): `n_unique` places of `n_keyframes` consecutive key frames
    (clouds in their own frame, key_leaf-filtered, with their true poses), then one key frame per candidate pair: a
    scan_leaf-filtered sweep taken in the middle of a place, carrying a drifted pose (offset <= 2 m, 5 deg) the way the
    latest key frame of the odometry does.  Returns dict(clouds, poses, scan_ids, center_ids, corrections):
    pair i aligns key frame scan_ids[i] (transformed by its pose) to the neighbourhood of key frame center_ids[i]."""

    def make():
        w = World(seed)
        out = {}
        for u in range(n_unique):
            base = 30 * u
            for k in range(n_keyframes):
                pose = trajectory_pose(base + k)
                sw = drop_invalid(cast_sweep(w, pose, frame=40_000 + base + k, n_beams=n_beams, n_azimuth=n_azimuth))
                out["kf%d_%d" % (u, k)] = numpy_voxel_downsample(sw, key_leaf)
                out["kfpose%d_%d" % (u, k)] = pose
            pose_s = trajectory_pose(base + n_keyframes // 2 + 0.4)
            sw = drop_invalid(cast_sweep(w, pose_s, frame=50_000 + u, n_beams=n_beams, n_azimuth=n_azimuth))
            out["scan%d" % u] = numpy_voxel_downsample(sw, scan_leaf)
            out["pose%d" % u] = pose_s
        return out

    d = _cached("loop_keyframes", (n_keyframes, n_beams, n_azimuth, scan_leaf, key_leaf, seed, n_unique, 1), make)
    clouds, poses = [], []
    for u in range(n_unique):
        for k in range(n_keyframes):
            clouds.append(d["kf%d_%d" % (u, k)])
            poses.append(d["kfpose%d_%d" % (u, k)].astype(np.float32))
    scan_ids, center_ids, corrections = [], [], []
    for i in range(n_pairs):
        u = i % n_unique
        rs = np.random.RandomState(1000 + i)
        dxy = rs.uniform(-1, 1, 2) * 2.0 / np.sqrt(2)
        yaw = np.radians(5.0) * rs.uniform(-1, 1)
        off = pose_matrix(dxy[0], dxy[1], yaw, z=0.0)
        clouds.append(d["scan%d" % u])
        poses.append((off @ d["pose%d" % u]).astype(np.float32))
        scan_ids.append(len(clouds) - 1)
        center_ids.append(u * n_keyframes + n_keyframes // 2)
        corrections.append(np.linalg.inv(off))
    return dict(clouds=clouds, poses=poses, scan_ids=scan_ids, center_ids=center_ids, corrections=corrections)


def rolling_map(n_points=20_000_000, seed=SEED):
    """cfg 3: a large rolling map of exactly `n_points` points: the cfg 0 local map (20 keyframes of the synthetic
    world) laid out again and again along the drive (60 m apart, alternate rows 35 m to the side, each copy with its own
    sub-voxel shift so that no two copies voxelise alike), plus the cfg 0 sweep and guess, which register against the
    first copy.  Returns dict(source, target, T_true, guess)."""
    d = ndt_scan_to_map(seed=seed)
    base = d["target"]
    n_copies = (n_points + len(base) - 1) // len(base)
    rs = np.random.RandomState((seed ^ 0x5EED) & 0x7FFFFFFF)
    out = np.empty((n_copies * len(base), 4), np.float32)
    for j in range(n_copies):
        shift = np.array([60.0 * (j // 2), 35.0 * (j % 2), 0.0], np.float32)
        if j:
            shift += rs.uniform(-0.5, 0.5, 3).astype(np.float32) * np.array([1, 1, 0.1], np.float32)
        blk = out[j * len(base):(j + 1) * len(base)]
        blk[:, :3] = base[:, :3] + shift
        blk[:, 3] = base[:, 3]
    return dict(source=d["source"], target=out[:n_points], T_true=d["T_true"], guess=d["guess"])
