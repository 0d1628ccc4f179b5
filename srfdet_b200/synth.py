"""Seeded synthetic inputs for parity tests and the bench (SURVEY.md 8d).

All generators run on the host with numpy.random.default_rng(seed) and return float32
numpy arrays, so the CPU oracle and the CUDA path see byte-identical inputs.
Geometry constants are the reference configs' (configs/nus/srfdet_voxel_nusc_L.py:6-13,
configs/kitti/srfdet_voxel_kitti_L.py:6-13, configs/waymo/srfdet_dvoxel_waymo_L.py:6-10).
"""
import math

import numpy as np

GEOM = {
    'nusc': dict(voxel_size=[0.075, 0.075, 0.2], pc_range=[-55.2, -55.2, -5.0, 55.2, 55.2, 3.0],
                 sparse_shape=[41, 1472, 1472], in_channels=5, n_points=300000,
                 max_points=10, max_voxels=160000),
    'kitti': dict(voxel_size=[0.05, 0.05, 0.1], pc_range=[0, -40, -3, 70.4, 40, 1],
                  sparse_shape=[41, 1600, 1408], in_channels=4, n_points=120000),
    'waymo': dict(voxel_size=[0.1, 0.1, 0.15], pc_range=[-76.8, -76.8, -2, 76.8, 76.8, 4],
                  sparse_shape=[41, 1536, 1536], in_channels=5, n_points=180000),
}


def _ring_cloud(rng, n, n_beams, elev_lo, elev_hi, az_lo, az_hi, max_range, sensor_h, n_boxes):
    """Surface-like spinning-LiDAR model: ~55 % ground returns of the downward beams (ring
    pattern, dense near the sensor), ~35 % returns on vertical facades, ~10 % on box-shaped
    objects.  Real scans are 2-D surfaces in 3-D, which is what sets the voxel counts per
    encoder level and the neighbours per voxel; uniformly scattered points would not."""
    n_obj = n // 10 if n_boxes else 0
    n_wall_target = int(n * 0.35)
    elevs = np.deg2rad(np.linspace(elev_lo, elev_hi, n_beams))
    # facades: random vertical rectangles, hit by the discrete beam set (horizontal scan lines)
    n_walls = 60
    wc = np.stack([rng.uniform(-0.8, 0.8, n_walls) * max_range, rng.uniform(-0.8, 0.8, n_walls) * max_range], 1)
    if az_lo >= -math.pi / 2 and az_hi <= math.pi / 2:
        wc[:, 0] = np.abs(wc[:, 0]) + 5.0
        wc[:, 1] *= 0.6
    wang = rng.uniform(0, math.pi, n_walls)
    wlen = rng.uniform(8, 40, n_walls)
    whgt = rng.uniform(3, 9, n_walls)
    m = 4 * n_wall_target
    wi = rng.integers(0, n_walls, m)
    t = rng.uniform(-0.5, 0.5, m) * wlen[wi]
    wx = wc[wi, 0] + t * np.cos(wang[wi])
    wy = wc[wi, 1] + t * np.sin(wang[wi])
    rr = np.hypot(wx, wy)
    we = rng.choice(elevs, m) + np.deg2rad(rng.uniform(-0.03, 0.03, m))
    wz = rr * np.tan(we)
    ok = (wz > -sensor_h + 0.1) & (wz < -sensor_h + whgt[wi]) & (rr < max_range) & (rr > 1.0)
    keep = np.nonzero(ok)[0][:n_wall_target]
    wx, wy, wz = wx[keep] + rng.normal(0, 0.01, len(keep)), wy[keep] + rng.normal(0, 0.01, len(keep)), wz[keep]
    n_wall = len(keep)
    n_gnd = n - n_obj - n_wall
    # ground: beams with negative elevation (ring pattern)
    down = elevs[elevs < -0.5 * np.pi / 180]
    e = rng.choice(down, n_gnd) + np.deg2rad(rng.uniform(-0.03, 0.03, n_gnd))
    az = rng.uniform(az_lo, az_hi, n_gnd)
    r = np.minimum(sensor_h / np.sin(-e), max_range)
    gx, gy = r * np.cos(e) * np.cos(az), r * np.cos(e) * np.sin(az)
    gz = -r * np.sin(-e) + rng.normal(0, 0.02, n_gnd)
    x = np.concatenate([gx, wx])
    y = np.concatenate([gy, wy])
    z = np.concatenate([gz, wz])
    if n_obj:
        bc = np.stack([rng.uniform(-0.6, 0.6, n_boxes) * max_range, rng.uniform(-0.6, 0.6, n_boxes) * max_range], 1)
        if az_lo >= -math.pi / 2 and az_hi <= math.pi / 2:
            bc[:, 0] = np.abs(bc[:, 0]) + 3.0
        which = rng.integers(0, n_boxes, n_obj)
        size = np.array([4.5, 1.9, 1.6])
        u = rng.uniform(-0.5, 0.5, (n_obj, 3)) * size
        face = rng.integers(0, 3, n_obj)
        u[np.arange(n_obj), face] = np.sign(u[np.arange(n_obj), face]) * size[face] / 2
        x = np.concatenate([x, bc[which, 0] + u[:, 0]])
        y = np.concatenate([y, bc[which, 1] + u[:, 1]])
        z = np.concatenate([z, -sensor_h + size[2] / 2 + u[:, 2]])
    perm = rng.permutation(n)          # interleave like a real scan (first-come order matters)
    return x[perm], y[perm], z[perm]


def _edge_points(rng, pts, pc_range, n_out_frac=0.03, n_face=16):
    """3 % of the points pushed outside the range and 16 points exactly on range faces."""
    n = pts.shape[0]
    k = int(n * n_out_frac)
    idx = rng.choice(n, k + n_face, replace=False)
    lo = np.array(pc_range[:3], np.float32)
    hi = np.array(pc_range[3:], np.float32)
    out = idx[:k]
    axis = rng.integers(0, 3, k)
    sign = rng.integers(0, 2, k)
    pts[out, axis] = np.where(sign == 1, hi[axis] + rng.uniform(0, 5, k), lo[axis] - rng.uniform(0, 5, k)).astype(np.float32)
    face = idx[k:]
    for t, i in enumerate(face):
        a = t % 3
        pts[i, a] = hi[a] if (t // 3) % 2 == 0 else lo[a]
    return pts


def cloud(kind, seed=0, n_points=None):
    """kind in {'nusc','kitti','waymo'} -> (N,C) float32 point cloud."""
    g = GEOM[kind]
    rng = np.random.default_rng(seed)
    n = int(n_points or g['n_points'])
    if kind == 'nusc':
        sweeps = 10
        x, y, z = _ring_cloud(rng, n, 32, -30.0, 10.0, -math.pi, math.pi, 60.0, 1.84, 40)
        sw = rng.integers(0, sweeps, n)
        x = x + 0.1 * sw  # per-sweep ego shift
        feats = np.stack([x, y, z, rng.integers(0, 256, n).astype(np.float64), 0.05 * sw], 1)
    elif kind == 'kitti':
        x, y, z = _ring_cloud(rng, n, 64, -24.8, 2.0, -math.pi / 4, math.pi / 4, 80.0, 1.73, 40)
        feats = np.stack([x, y, z, rng.uniform(0, 1, n)], 1)
    elif kind == 'waymo':
        x, y, z = _ring_cloud(rng, n, 64, -17.6, 2.4, -math.pi, math.pi, 75.0, 1.8, 40)
        feats = np.stack([x, y, z, rng.uniform(0, 1, n), rng.uniform(0, 1, n)], 1)
    else:
        raise KeyError(kind)
    pts = feats.astype(np.float32)
    return np.ascontiguousarray(_edge_points(rng, pts, g['pc_range']))


def dense_cloud(kind, seed, n_points, extent=6.0):
    """Small-extent cloud: many points per voxel (exercises max_points / max_voxels)."""
    g = GEOM[kind]
    rng = np.random.default_rng(seed)
    c = g['in_channels']
    pts = rng.uniform(-extent, extent, (n_points, c)).astype(np.float32)
    pts[:, 2] = rng.uniform(-1.0, 0.5, n_points)
    if kind == 'kitti':
        pts[:, 0] = np.abs(pts[:, 0]) + 1.0
    return np.ascontiguousarray(pts)


def proposals(seed, n=900, dims=10, batch=1):
    """(B,n,dims): centres U[0,1]^3, log-sizes N(log[1.9,4.6,1.7],0.3^2), yaw U[-pi,pi]."""
    rng = np.random.default_rng(seed)
    b = np.zeros((batch, n, dims), np.float32)
    b[..., :3] = rng.uniform(0, 1, (batch, n, 3))
    b[..., 3:6] = np.log(np.array([1.9, 4.6, 1.7])) + 0.3 * rng.standard_normal((batch, n, 3))
    yaw = rng.uniform(-math.pi, math.pi, (batch, n))
    b[..., 6] = np.sin(yaw)
    b[..., 7] = np.cos(yaw)
    return b


def lidar2img(n_cam=6, batch=1, yaw_offsets=None):
    """nuScenes-like projection matrices built by the recipe of
    datasets/nuscenes_dataset.py:53-65: lidar2img = viewpad(K) @ [R^T | -R^T t]^T.
    yaw_offsets: one angle (radians) per sample that turns its whole camera rig about the LiDAR z axis, so the
    samples of a batch see different projections; None: every sample has the same rig."""
    if yaw_offsets is not None:
        assert len(yaw_offsets) == batch
        base = lidar2img(n_cam, 1)[0].astype(np.float64)
        out = np.zeros((batch, n_cam, 4, 4), np.float32)
        for b, a in enumerate(yaw_offsets):
            rz = np.eye(4)      # a rig turned by a sees the LiDAR frame turned by -a
            rz[:2, :2] = [[math.cos(a), math.sin(a)], [-math.sin(a), math.cos(a)]]
            out[b] = (base @ rz).astype(np.float32)
        return out
    yaws = np.deg2rad([0.0, 55.0, -55.0, 110.0, -110.0, 180.0])[:n_cam]
    K = np.array([[1266.0, 0, 816.0], [0, 1266.0, 491.0], [0, 0, 1.0]])
    out = np.zeros((batch, n_cam, 4, 4), np.float32)
    for c, yaw in enumerate(yaws):
        # camera axes in lidar frame: z forward, x right, y down
        fwd = np.array([math.cos(yaw), math.sin(yaw), 0.0])
        right = np.array([math.sin(yaw), -math.cos(yaw), 0.0])
        down = np.array([0.0, 0.0, -1.0])
        R = np.stack([right, down, fwd], 0)           # lidar -> cam rotation
        t = np.array([0.0, 0.0, 1.5 - 1.84])          # camera position in lidar frame
        rt = np.eye(4)
        rt[:3, :3] = R
        rt[:3, 3] = -R @ t
        vp = np.eye(4)
        vp[:3, :3] = K
        out[:, c] = (vp @ rt).astype(np.float32)
    return out


def feature_pyramid(seed, channels, base_hw, n_levels=4, lead=(1,)):
    """N(0,1) fp32 maps lead+(C,H/2^l,W/2^l) standing in for FPN outputs (the dense
    backbones are outside the hot path, SURVEY.md 8d)."""
    rng = np.random.default_rng(seed)
    h, w = base_hw
    out = []
    for _ in range(n_levels):
        out.append(rng.standard_normal(tuple(lead) + (channels, h, w), dtype=np.float32))
        h, w = (h + 1) // 2, (w + 1) // 2
    return out


def hash_field(shape, seed):
    """Deterministic pseudo-random fp32 field in [-1, 1) built from integer hashing only
    (bit-identical on every machine, so fixtures need not store it)."""
    idx = np.indices(shape, dtype=np.uint64)
    primes = [np.uint64(p) for p in (73856093, 19349663, 83492791, 2654435761, 40503, 2246822519)]
    h = np.full(shape, np.uint64(seed * 1000003 + 12345), np.uint64)
    for d in range(len(shape)):
        h = (h ^ (idx[d] * primes[d % len(primes)])) * np.uint64(0x9E3779B97F4A7C15)
        h ^= h >> np.uint64(29)
    return ((h >> np.uint64(40)) % np.uint64(4096)).astype(np.float32) / np.float32(2048.0) - np.float32(1.0)
