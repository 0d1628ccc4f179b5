"""Reference for the multi-sweep point input (srf_merge_sweeps / plugin/points.py), restating mmdet3d 1.0.0rc6
(datasets/pipelines/loading.py LoadPointsFromFile, LoadPointsFromMultiSweeps; transforms_3d.py PointsRangeFilter;
core/points/base_points.py in_range_3d).  Nothing is vendored.

merge():          numpy with the rounding spelled out: every product and sum of the rotation in float64 in the order
                  ((x R_i0 + y R_i1) + z R_i2), rounded to float32, then + t in float64 rounded to float32.  The kernel
                  must equal it bit for bit.
LiteralMultiSweeps / literal_range_filter: a line-by-line transcription of the rc6 __call__ bodies over a minimal
                  stand-in for LiDARPoints (a torch tensor), with numpy's BLAS matmul, whose summation order is its own:
                  values within 1 float32 ulp of merge().
Samples are info dicts (lidar_path, timestamp in us, sweeps=[dict(data_path, sensor2lidar_rotation,
sensor2lidar_translation, timestamp)]); arrays stand in for the files.
"""
import numpy as np
import torch


def load(src, load_dim):
    raw = np.fromfile(src, dtype=np.float32) if isinstance(src, str) else np.asarray(src, np.float32)
    return raw.reshape(-1, load_dim).copy()


def rigid(xyz, rot, trans):
    """float32 (n, 3), float64 R (3, 3), t (3,) -> float32, numpy's two-step rounding with a fixed summation order."""
    x, y, z = (xyz[:, j].astype(np.float64) for j in range(3))
    rot = np.asarray(rot, np.float64)
    trans = np.asarray(trans, np.float64)
    out = np.empty_like(xyz)
    for i in range(3):
        r = ((x * rot[i, 0] + y * rot[i, 1]) + z * rot[i, 2]).astype(np.float32)
        out[:, i] = (r.astype(np.float64) + trans[i]).astype(np.float32)
    return out


def remove_close(points, radius=1.0):
    keep = ~((np.abs(points[:, 0]) < np.float32(radius)) & (np.abs(points[:, 1]) < np.float32(radius)))
    return points[keep]


def range_filter(points, pcr):
    lo = np.asarray(pcr[:3], np.float32)
    hi = np.asarray(pcr[3:], np.float32)
    keep = np.all((points[:, :3] > lo) & (points[:, :3] < hi), axis=1)
    return points[keep]


def merge(sample, load_dim=5, use_dim=5, sweeps=None, pcr=None, choices=None):
    """sweeps: LoadPointsFromMultiSweeps arguments (sweeps_num, load_dim, use_dim, pad_empty_sweeps, remove_close) or
    None; choices: the sweep indices read (default: the first min(len, sweeps_num)).  -> (n, len(use_dim)) float32."""
    use = list(range(use_dim)) if isinstance(use_dim, int) else list(use_dim)
    key = load(sample['lidar_path'], load_dim)[:, use]
    if sweeps is not None:
        key[:, 4] = 0
        parts = [key]
        ts = sample['timestamp'] / 1e6
        if sweeps.get('pad_empty_sweeps', False) and len(sample['sweeps']) == 0:
            for _ in range(sweeps['sweeps_num']):
                parts.append(remove_close(key) if sweeps.get('remove_close', False) else key)
        else:
            if choices is None:
                choices = range(min(len(sample['sweeps']), sweeps['sweeps_num']))
            for idx in choices:
                sw = sample['sweeps'][idx]
                p = load(sw['data_path'], sweeps['load_dim'])
                if sweeps.get('remove_close', False):
                    p = remove_close(p)
                p[:, :3] = rigid(p[:, :3], sw['sensor2lidar_rotation'], sw['sensor2lidar_translation'])
                p[:, 4] = ts - sw['timestamp'] / 1e6
                parts.append(p)
        key = np.concatenate(parts, 0)[:, list(sweeps['use_dim'])]
    return range_filter(key, pcr) if pcr is not None else key


# ------------------------------------------------------------------------------------- literal transcription
class _Points:
    """The parts of mmdet3d's LiDARPoints the rc6 __call__ bodies use."""

    def __init__(self, tensor):
        self.tensor = torch.as_tensor(tensor, dtype=torch.float32)

    def new_point(self, data):
        return _Points(torch.as_tensor(np.asarray(data), dtype=torch.float32).clone())

    def cat(self, points_list):
        return _Points(torch.cat([p.tensor for p in points_list], dim=0))

    def __getitem__(self, item):
        if isinstance(item, np.ndarray):
            item = torch.from_numpy(item)
        return _Points(self.tensor[item])

    def in_range_3d(self, point_range):
        return ((self.tensor[:, 0] > point_range[0]) & (self.tensor[:, 1] > point_range[1])
                & (self.tensor[:, 2] > point_range[2]) & (self.tensor[:, 0] < point_range[3])
                & (self.tensor[:, 1] < point_range[4]) & (self.tensor[:, 2] < point_range[5]))


def literal_load_points_from_file(pts_filename, load_dim, use_dim):
    use_dim = list(range(use_dim)) if isinstance(use_dim, int) else use_dim
    points = load(pts_filename, load_dim)
    points = points.reshape(-1, load_dim)
    points = points[:, use_dim]
    return _Points(points)


class LiteralMultiSweeps:
    def __init__(self, sweeps_num=10, load_dim=5, use_dim=[0, 1, 2, 4], pad_empty_sweeps=False, remove_close=False,
                 test_mode=False):
        self.load_dim = load_dim
        self.sweeps_num = sweeps_num
        self.use_dim = use_dim
        self.pad_empty_sweeps = pad_empty_sweeps
        self.remove_close = remove_close
        self.test_mode = test_mode

    def _load_points(self, pts_filename):
        return load(pts_filename, self.load_dim).reshape(-1)

    def _remove_close(self, points, radius=1.0):
        if isinstance(points, np.ndarray):
            points_numpy = points
        else:
            points_numpy = points.tensor.numpy()
        x_filt = np.abs(points_numpy[:, 0]) < radius
        y_filt = np.abs(points_numpy[:, 1]) < radius
        not_close = np.logical_not(np.logical_and(x_filt, y_filt))
        return points[not_close]

    def __call__(self, results):
        points = results['points']
        points.tensor[:, 4] = 0
        sweep_points_list = [points]
        ts = results['timestamp']
        if self.pad_empty_sweeps and len(results['sweeps']) == 0:
            for i in range(self.sweeps_num):
                if self.remove_close:
                    sweep_points_list.append(self._remove_close(points))
                else:
                    sweep_points_list.append(points)
        else:
            if len(results['sweeps']) <= self.sweeps_num:
                choices = np.arange(len(results['sweeps']))
            elif self.test_mode:
                choices = np.arange(self.sweeps_num)
            else:
                choices = np.random.choice(len(results['sweeps']), self.sweeps_num, replace=False)
            for idx in choices:
                sweep = results['sweeps'][idx]
                points_sweep = self._load_points(sweep['data_path'])
                points_sweep = np.copy(points_sweep).reshape(-1, self.load_dim)
                if self.remove_close:
                    points_sweep = self._remove_close(points_sweep)
                sweep_ts = sweep['timestamp'] / 1e6
                points_sweep[:, :3] = points_sweep[:, :3] @ sweep['sensor2lidar_rotation'].T
                points_sweep[:, :3] += sweep['sensor2lidar_translation']
                points_sweep[:, 4] = ts - sweep_ts
                points_sweep = points.new_point(points_sweep)
                sweep_points_list.append(points_sweep)

        points = points.cat(sweep_points_list)
        points = points[:, self.use_dim]
        results['points'] = points
        return results


def literal_range_filter(points, point_cloud_range):
    pcr = np.array(point_cloud_range, dtype=np.float32)
    points_mask = points.in_range_3d(pcr)
    return points[points_mask]


def literal_pipeline(sample, load_dim=5, use_dim=5, sweeps=None, pcr=None):
    """LoadPointsFromFile -> LoadPointsFromMultiSweeps -> PointsRangeFilter as the rc6 dataset runs them
    (results['timestamp'] = info['timestamp'] / 1e6, NuScenesDataset.get_data_info).  -> float32 numpy."""
    results = dict(points=literal_load_points_from_file(sample['lidar_path'], load_dim, use_dim),
                   timestamp=sample['timestamp'] / 1e6, sweeps=sample['sweeps'])
    if sweeps is not None:
        results = LiteralMultiSweeps(**sweeps)(results)
    pts = results['points']
    if pcr is not None:
        pts = literal_range_filter(pts, pcr)
    return pts.tensor.numpy()


# ------------------------------------------------------------------------------------- synthetic samples
def random_rotation(rng, max_tilt=0.05):
    """Rigid rotation: a yaw anywhere and a small roll / pitch (a LiDAR moving on a road)."""
    a, b, c = rng.uniform(-np.pi, np.pi), rng.uniform(-max_tilt, max_tilt), rng.uniform(-max_tilt, max_tilt)
    rz = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
    ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    rx = np.array([[1, 0, 0], [0, np.cos(c), -np.sin(c)], [0, np.sin(c), np.cos(c)]])
    return rz @ ry @ rx


NUSC_RANGE = [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]


def edge_points(pcr=NUSC_RANGE):
    """Points on the close-removal square (|x| or |y| exactly 1) and exactly on every face of the range."""
    lo, hi = np.float32(pcr[:3]), np.float32(pcr[3:])
    pts = [[1.0, 0.5, 0.0], [-1.0, 0.2, 0.0], [0.5, 1.0, 0.0], [0.3, -1.0, 0.0], [1.0, 1.0, 0.0], [0.99, -0.99, 0.0],
           [np.nextafter(np.float32(1), np.float32(0)), 0.0, 0.0]]
    for j in range(3):
        for v in (lo[j], hi[j], np.nextafter(lo[j], hi[j]), np.nextafter(hi[j], lo[j])):
            p = [5.0, 5.0, 0.0]
            p[j] = v
            pts.append(p)
    return np.asarray(pts, np.float32)


def cloud(rng, n, load_dim=5, span=60.0):
    xyz = np.stack([rng.uniform(-span, span, n), rng.uniform(-span, span, n), rng.uniform(-6.0, 4.0, n)], 1)
    extra = np.stack([rng.integers(0, 256, n).astype(np.float64), rng.integers(0, 32, n).astype(np.float64)]
                     + [rng.normal(size=n) for _ in range(load_dim - 5)], 1)
    return np.concatenate([xyz, extra], 1).astype(np.float32)


def make_sample(rng, n_key, n_sweeps, load_dim=5, edges=True):
    """Key frame of n_key points and one sweep per entry of n_sweeps, random rigid poses, timestamps in us decreasing
    by about 50 ms.  With edges: edge_points() in the key frame; in the first sweep under an identity rotation and a
    translation of (2, 0, 0), points that land exactly on the range faces, and raw points on the close square."""
    ts = int(1533151603547590 + rng.integers(0, 10 ** 9))
    key = cloud(rng, n_key, load_dim)
    e = edge_points()
    if edges:
        ek = np.zeros((len(e), load_dim), np.float32)
        ek[:, :3] = e
        ek[:, 3] = 7.0
        key = np.concatenate([key[: n_key // 2], ek, key[n_key // 2:]], 0)
    sweeps = []
    for i, n in enumerate(n_sweeps):
        pts = cloud(rng, n, load_dim)
        rot, trans = random_rotation(rng), rng.normal(scale=3.0, size=3)
        if edges and i == 0:
            rot, trans = np.eye(3), np.array([2.0, 0.0, 0.0])
            onface = e.copy()
            onface[:, 0] = (e[:, 0].astype(np.float64) - 2.0).astype(np.float32)   # exact: x + 2 == e.x in float32
            es = np.zeros((len(e), load_dim), np.float32)
            es[:, :3] = onface
            es[:, 3] = 9.0
            close = np.zeros((len(e), load_dim), np.float32)
            close[:, :3] = e
            pts = np.concatenate([es, close, pts], 0)
        sweeps.append(dict(data_path=pts.reshape(-1), sensor2lidar_rotation=rot, sensor2lidar_translation=trans,
                           timestamp=ts - 50000 * (i + 1) - int(rng.integers(0, 2000))))
    return dict(lidar_path=key.reshape(-1), timestamp=ts, sweeps=sweeps)
