"""Point input of a reference config's test pipeline on the GPU: nuScenes sweeps in, fixed-capacity clouds out.

mmdet3d 1.0.0rc6's LoadPointsFromFile, LoadPointsFromMultiSweeps and PointsRangeFilter (restated, nothing vendored)
become one device stage (srf_merge_sweeps, csrc/sweeps.cu).  Its clouds have a fixed number of rows: the valid points
first, in the reference's order, then NaN rows, which both voxelizers drop as out of range.  A padded cloud therefore
voxelizes exactly like the compact one, and every frame of a sequence has the same shape, so SRFDet.infer(use_graph=True)
captures one graph for the whole sequence.

    loader = MultiSweepLoader.from_config('srfdet_voxel_nusc_L.py', batch_size=1, max_points=40000)
    for info in load_nuscenes_infos('nuscenes_infos_val.pkl', data_root='data/nuscenes'):
        loader.stage([info])
        clouds, counts = loader()
        det.infer(clouds)
"""
import _compat_pickle
import collections
import ctypes
import io
import os
import pickle

import numpy as np
import torch

from .. import _lib as L

PointSteps = collections.namedtuple('PointSteps', ['load_dim', 'use_dim', 'sweeps', 'point_cloud_range'])
PointSteps.__doc__ = """The point steps of a test pipeline: LoadPointsFromFile's load_dim / use_dim (a list), the
LoadPointsFromMultiSweeps settings (a dict with all its arguments, or None) and PointsRangeFilter's range (or None)."""

_SWEEP_DEFAULTS = dict(sweeps_num=10, load_dim=5, use_dim=[0, 1, 2, 4], pad_empty_sweeps=False, remove_close=False,
                       test_mode=False)
# steps that do not touch the points: image loading / preprocessing and the final formatting
_IGNORED = ('LoadMultiViewImageFromFiles', 'NormalizeMultiviewImage', 'PadMultiViewImage', 'ResizeMultiview3D',
            'ResizeCropFlipImage', 'PhotoMetricDistortionMultiViewImage', 'LoadImageFromFile', 'Normalize', 'Pad',
            'Resize', 'DefaultFormatBundle3D', 'DefaultFormatBundle', 'Collect3D', 'Collect')


def _as_dims(use_dim):
    return list(range(use_dim)) if isinstance(use_dim, int) else [int(d) for d in use_dim]


def _is_identity_rot_scale_trans(step):
    # mmdet3d 1.0.0rc6 GlobalRotScaleTrans defaults: rot_range +-pi/4, scale_ratio_range [0.95, 1.05]
    rot = step.get('rot_range', [-0.78539816, 0.78539816])
    rot = [-rot, rot] if isinstance(rot, (int, float)) else list(rot)
    scale = list(step.get('scale_ratio_range', [0.95, 1.05]))
    trans = step.get('translation_std', [0, 0, 0])
    trans = [trans] * 3 if isinstance(trans, (int, float)) else list(trans)
    return rot == [0, 0] and scale == [1, 1] and trans == [0, 0, 0] and not step.get('shift_height', False)


def _point_step(step, acc):
    """LoadPointsFromFile / LoadPointsFromMultiSweeps / PointsRangeFilter into acc ('load', 'sweeps', 'pcr');
    -> True when the step was one of them."""
    t = step['type']
    if t == 'LoadPointsFromFile':
        if step.get('shift_height', False) or step.get('use_color', False):
            raise NotImplementedError('LoadPointsFromFile: shift_height / use_color are not supported')
        acc['load'] = (int(step.get('load_dim', 6)), _as_dims(step.get('use_dim', [0, 1, 2])))
    elif t == 'LoadPointsFromMultiSweeps':
        sweeps = {k: step.get(k, v) for k, v in _SWEEP_DEFAULTS.items()}
        sweeps['use_dim'] = _as_dims(sweeps['use_dim'])
        acc['sweeps'] = sweeps
    elif t == 'PointsRangeFilter':
        acc['pcr'] = [float(v) for v in step['point_cloud_range']]
    else:
        return False
    return True


def _point_steps(acc):
    load, sweeps, pcr = acc['load'], acc['sweeps'], acc['pcr']
    if load is None:
        raise ValueError('the test pipeline has no LoadPointsFromFile step')
    if load[1][:3] != [0, 1, 2] or (sweeps and sweeps['use_dim'][:3] != [0, 1, 2]):
        raise NotImplementedError('use_dim must start with the coordinates 0, 1, 2')
    if sweeps and len(load[1]) != sweeps['load_dim']:
        raise ValueError(f'LoadPointsFromFile keeps {len(load[1])} columns but LoadPointsFromMultiSweeps loads '
                         f'{sweeps["load_dim"]}: the reference concatenates them, so they must agree')
    if sweeps and sweeps['load_dim'] < 5:
        raise ValueError('LoadPointsFromMultiSweeps writes the time lag into column 4: load_dim must be >= 5')
    return PointSteps(load[0], load[1], sweeps, pcr)


def parse_test_pipeline(pipeline):
    """-> PointSteps of a config's `test_pipeline` (a list of step dicts).  MultiScaleFlipAug3D's transforms are searched
    too.  Steps that leave the points bit-identical at test time are accepted: MultiScaleFlipAug3D(flip=False,
    pts_scale_ratio=1), GlobalRotScaleTrans(rot_range=[0, 0], scale_ratio_range=[1, 1], translation_std=[0, 0, 0]) and
    RandomFlip3D inside MultiScaleFlipAug3D(flip=False).  Image and formatting steps are ignored; any other step or
    setting raises NotImplementedError naming it.  Test-time augmentation: parse_test_augmentations."""
    acc = dict(load=None, sweeps=None, pcr=None)

    def walk(steps, in_noflip_aug):
        for step in steps:
            t = step['type']
            if _point_step(step, acc):
                continue
            if t == 'MultiScaleFlipAug3D':
                ratio = step.get('pts_scale_ratio', 1)
                ratio = list(ratio) if isinstance(ratio, (list, tuple)) else [ratio]
                if step.get('flip', False) or ratio != [1]:
                    raise NotImplementedError('MultiScaleFlipAug3D: only flip=False, pts_scale_ratio=1 (no test-time '
                                              f'augmentation) is supported, got flip={step.get("flip")}, '
                                              f'pts_scale_ratio={step.get("pts_scale_ratio")}')
                walk(step['transforms'], True)
            elif t == 'GlobalRotScaleTrans':
                if not _is_identity_rot_scale_trans(step):
                    raise NotImplementedError(f'GlobalRotScaleTrans: only the identity (rot_range=[0, 0], scale_ratio_range='
                                              f'[1, 1], translation_std=[0, 0, 0]) is supported, got {step}')
            elif t == 'RandomFlip3D':
                if not in_noflip_aug:
                    raise NotImplementedError('RandomFlip3D is supported only inside MultiScaleFlipAug3D(flip=False)')
            elif t not in _IGNORED:
                raise NotImplementedError(f'{t}: this test-pipeline step is not supported by the point loader')

    walk(pipeline, False)
    return _point_steps(acc)


IDENTITY_VIEW = (1.0, False, False)


class PointAugmentation(collections.namedtuple('PointAugmentation', ['steps', 'views', 'range_position'])):
    """Test-time augmentation of a config's `test_pipeline` (parse_test_augmentations).
    steps: the single-view PointSteps (point_cloud_range: the PointsRangeFilter's range wherever it sits);
    views: [(pcd_scale_factor, horizontal flip, vertical flip)] in MultiScaleFlipAug3D's order, duplicates included;
    range_position: 'before' or 'after' the augmentation, None without a range filter."""
    __slots__ = ()

    @property
    def loader_steps(self):
        """Steps of the point loader: without the range filter when it runs after the augmentation
        (srf_augment_points applies it to each view)."""
        return self.steps._replace(point_cloud_range=None) if self.range_position == 'after' else self.steps

    @property
    def view_range(self):
        """The range srf_augment_points tests each view against, or None."""
        return self.steps.point_cloud_range if self.range_position == 'after' else None

    @property
    def augments(self):
        """The reference runs aug_test (more than one view, or one that changes the points)."""
        return list(self.views) != [IDENTITY_VIEW]


def distinct_views(views):
    """The distinct views in first-occurrence order."""
    return list(dict.fromkeys((float(s), bool(h), bool(v)) for s, h, v in views))


def parse_test_augmentations(pipeline):
    """-> PointAugmentation of a config's `test_pipeline`, with mmdet3d 1.0.0rc6's MultiScaleFlipAug3D expansion: loops
    img_scale -> pts_scale_ratio (a list) -> flip in [False, True] if flip else [False] -> pcd_horizontal_flip in
    [False, True] if flip and pcd_horizontal_flip else [False] -> the same for pcd_vertical_flip -> flip_direction.
    RandomFlip3D with sync_2d=True (its default) flips horizontally when `flip` and never vertically; with
    sync_2d=False it takes the wrapper's pcd flags.  Inside the wrapper GlobalRotScaleTrans must have the identity
    rotation and translation (its scale_ratio_range is ignored: the wrapper sets pcd_scale_factor).  NotImplementedError
    for scale ratios other than 1 without GlobalRotScaleTrans and for flip=True without RandomFlip3D (the reference would
    map boxes back that were never augmented), and for the steps parse_test_pipeline refuses."""
    acc = dict(load=None, sweeps=None, pcr=None)
    aug, state = None, dict(range_position=None, augmenting_seen=False, scale=False, flip3d=None)

    def walk(steps, in_aug):
        nonlocal aug
        for step in steps:
            t = step['type']
            if _point_step(step, acc):
                if t == 'PointsRangeFilter':
                    state['range_position'] = 'after' if state['augmenting_seen'] else 'before'
                continue
            if t == 'MultiScaleFlipAug3D':
                if aug is not None:
                    raise NotImplementedError('MultiScaleFlipAug3D: one wrapper per test pipeline is supported')
                aug = step
                walk(step['transforms'], True)
            elif t == 'GlobalRotScaleTrans':
                if not in_aug:
                    if not _is_identity_rot_scale_trans(step):
                        raise NotImplementedError(f'GlobalRotScaleTrans outside MultiScaleFlipAug3D: only the identity is '
                                                  f'supported, got {step}')
                    continue
                if not _is_identity_rot_scale_trans(dict(step, scale_ratio_range=[1, 1])):
                    raise NotImplementedError(f'GlobalRotScaleTrans: only the identity rotation and translation (rot_range='
                                              f'[0, 0], translation_std=[0, 0, 0]) are supported, got {step}')
                state['scale'] = state['augmenting_seen'] = True
            elif t == 'RandomFlip3D':
                if not in_aug:
                    raise NotImplementedError('RandomFlip3D is supported only inside MultiScaleFlipAug3D')
                state['flip3d'] = step
                state['augmenting_seen'] = True
            elif t not in _IGNORED:
                raise NotImplementedError(f'{t}: this test-pipeline step is not supported by the point loader')

    walk(pipeline, False)
    steps = _point_steps(acc)
    if aug is None:
        return PointAugmentation(steps, [IDENTITY_VIEW], state['range_position'])
    ratio = aug.get('pts_scale_ratio', 1)
    ratios = [float(r) for r in ratio] if isinstance(ratio, (list, tuple)) else [float(ratio)]
    flip = bool(aug.get('flip', False))
    if any(r != 1 for r in ratios) and not state['scale']:
        raise NotImplementedError(f'MultiScaleFlipAug3D(pts_scale_ratio={ratio}) without GlobalRotScaleTrans in its '
                                  'transforms: the points would not be scaled while the boxes are mapped back')
    if flip and state['flip3d'] is None:
        raise NotImplementedError('MultiScaleFlipAug3D(flip=True) without RandomFlip3D in its transforms: the points would '
                                  'not be flipped while the boxes are mapped back')
    img_scale, direction = aug.get('img_scale'), aug.get('flip_direction', 'horizontal')
    n_img = len(img_scale) if isinstance(img_scale, list) else 1
    n_dir = len(direction) if isinstance(direction, list) else 1
    hs = [False, True] if flip and aug.get('pcd_horizontal_flip', False) else [False]
    vs = [False, True] if flip and aug.get('pcd_vertical_flip', False) else [False]
    sync_2d = state['flip3d'] is None or state['flip3d'].get('sync_2d', True)
    views = [(s, f, False) if sync_2d else (s, h, v)
             for _ in range(n_img) for s in ratios for f in ([False, True] if flip else [False]) for h in hs for v in vs
             for _ in range(n_dir)]
    return PointAugmentation(steps, views, state['range_position'])


def choose_sweeps(n_sweeps, sweeps_num, test_mode):
    """Indices of the sweeps LoadPointsFromMultiSweeps reads (rc6): all when there are at most sweeps_num, else the first
    sweeps_num in test_mode, else np.random.choice(n_sweeps, sweeps_num, replace=False) (numpy's global generator)."""
    if n_sweeps <= sweeps_num:
        return list(range(n_sweeps))
    if test_mode:
        return list(range(sweeps_num))
    return [int(i) for i in np.random.choice(n_sweeps, sweeps_num, replace=False)]


# ---------------------------------------------------------------------------------------------- nuScenes infos
class _InfoUnpickler(pickle.Unpickler):
    """Builtin containers / scalars and numpy array, dtype and scalar reconstruction (numpy 1.x and 2.x module paths);
    every other global is refused, so a crafted file cannot call anything."""
    _ALLOWED = {
        ('builtins', n) for n in ('dict', 'list', 'tuple', 'set', 'frozenset', 'str', 'bytes', 'bytearray', 'int',
                                  'float', 'complex', 'bool', 'slice')
    } | {(m, n) for m in ('numpy.core.multiarray', 'numpy._core.multiarray') for n in ('_reconstruct', 'scalar')} | {
        ('numpy', 'ndarray'), ('numpy', 'dtype'),
        ('_codecs', 'encode'),        # protocol-2 pickles carry numpy's raw bytes as latin-1 text through it
    }

    def find_class(self, module, name):
        if (module, name) in _compat_pickle.NAME_MAPPING:       # protocol < 3: Python 2 names, as pickle maps them
            module, name = _compat_pickle.NAME_MAPPING[(module, name)]
        module = _compat_pickle.IMPORT_MAPPING.get(module, module)
        if (module, name) in self._ALLOWED:
            return super().find_class(module, name)
        raise pickle.UnpicklingError(f'nuScenes infos: refusing to load {module}.{name}')


def _reroot(path, data_root):
    if data_root is None:
        return path
    parts = path.replace('\\', '/').split('/')
    for anchor in ('samples', 'sweeps'):
        if anchor in parts:
            return os.path.join(data_root, *parts[parts.index(anchor):])
    return path if os.path.isabs(path) else os.path.join(data_root, path)


def load_nuscenes_infos(path, data_root=None):
    """Read mmdet3d's nuscenes_infos_*.pkl (dict(infos=[...], metadata=...) or a bare list) with a restricted unpickler.
    -> list of dict(lidar_path, timestamp, sweeps=[dict(data_path, sensor2lidar_rotation, sensor2lidar_translation,
    timestamp)]).  data_root: paths are re-rooted at it from their `samples/` or `sweeps/` component (the nuScenes
    directory layout); other relative paths are joined to it."""
    with open(path, 'rb') as f:
        data = _InfoUnpickler(io.BytesIO(f.read())).load()
    infos = data['infos'] if isinstance(data, dict) else data
    out = []
    for info in infos:
        sweeps = [dict(data_path=_reroot(s['data_path'], data_root),
                       sensor2lidar_rotation=np.asarray(s['sensor2lidar_rotation'], np.float64),
                       sensor2lidar_translation=np.asarray(s['sensor2lidar_translation'], np.float64),
                       timestamp=s['timestamp']) for s in info.get('sweeps', [])]
        out.append(dict(lidar_path=_reroot(info['lidar_path'], data_root), timestamp=info['timestamp'], sweeps=sweeps))
    return out


# ---------------------------------------------------------------------------------------------- loader
def _read_points(src, load_dim):
    """A file path (raw float32) or an array standing in for one -> (n, load_dim) float32."""
    raw = np.fromfile(src, dtype=np.float32) if isinstance(src, (str, os.PathLike)) else np.asarray(src, np.float32)
    if raw.size % load_dim:
        raise ValueError(f'{src if isinstance(src, (str, os.PathLike)) else "array"}: {raw.size} float32 values are not '
                         f'a multiple of load_dim {load_dim}')
    return raw.reshape(-1, load_dim)


class MultiSweepLoader:
    """Fixed-capacity device staging of B samples (one key frame + sweeps_num sweeps each, at most max_points points per
    file) and the merge kernel over it.

    stage(samples): reads the files on the host (ValueError when one exceeds max_points: nothing is cut), then copies
    each file, the counts, the poses and the time lags host -> device with non-blocking copies from pinned memory; no
    synchronisation.  A stage waits only for the copies of the previous stage before it reuses the pinned buffers.
    __call__(): runs the kernel -> (B clouds (capacity, n_cols) float32, counts (B,) int32 device); rows past a count are
    NaN.  The clouds live in the loader's buffers, which the next call overwrites.
    A sample is an info dict (load_nuscenes_infos); arrays may stand in for the lidar_path / data_path files."""

    def __init__(self, steps, batch_size=1, max_points=40000, device='cuda'):
        self.steps = steps
        self.batch_size, self.max_points, self.device = int(batch_size), int(max_points), torch.device(device)
        sw = steps.sweeps
        self.n_sweeps = int(sw['sweeps_num']) if sw else 0
        self.n_src = 1 + self.n_sweeps
        if self.n_src > L.SWEEP_MAX_SOURCES:
            raise ValueError(f'sweeps_num {self.n_sweeps}: at most {L.SWEEP_MAX_SOURCES - 1} sweeps are supported')
        self.width = len(steps.use_dim)           # row width of every staged file (key frame after its use_dim)
        self.cols = list(sw['use_dim']) if sw else list(range(self.width))
        if max(self.cols) >= self.width or len(self.cols) > L.SWEEP_MAX_COLS:
            raise ValueError(f'output columns {self.cols} do not fit rows of {self.width} values')
        self.n_cols = len(self.cols)
        self.capacity = self.n_src * self.max_points
        self._dev = None
        self._copied = None

    @classmethod
    def from_config(cls, path_or_cfg, **kwargs):
        """From a config file (plain Python) or its namespace dict: the point steps of its `test_pipeline`."""
        from .registry import load_config
        cfg = load_config(path_or_cfg) if isinstance(path_or_cfg, (str, os.PathLike)) else path_or_cfg
        if 'test_pipeline' not in cfg:
            raise ValueError('the config has no test_pipeline: the point loader reads its steps from there')
        return cls(parse_test_pipeline(cfg['test_pipeline']), **kwargs)

    # ------------------------------------------------------------------ host side
    def read(self, samples):
        """Host part of stage(), no device access: -> (files: per sample one (n, width) array per source, None where a
        padded empty sweep reads the key frame again; flags, counts (B, S), poses (B, S, 12), time lags (B, S))."""
        if len(samples) != self.batch_size:
            raise ValueError(f'expected {self.batch_size} samples, got {len(samples)}')
        st, sw = self.steps, self.steps.sweeps
        B, S = self.batch_size, self.n_src
        counts = np.zeros((B, S), np.int32)
        poses = np.zeros((B, S, 12), np.float64)
        lags = np.zeros((B, S), np.float32)
        files, flags = [], np.zeros((B, S), np.int32)
        close = L.SWEEP_REMOVE_CLOSE if sw and sw['remove_close'] else 0
        for b, smp in enumerate(samples):
            key = np.ascontiguousarray(_read_points(smp['lidar_path'], st.load_dim)[:, st.use_dim])
            self._check_cap(key, smp['lidar_path'])
            row = [key]
            counts[b, 0] = key.shape[0]
            flags[b, 0] = L.SWEEP_TIME_LAG if sw else 0          # the key frame's time lag is 0
            if sw:
                ts = smp['timestamp'] / 1e6
                if sw['pad_empty_sweeps'] and len(smp['sweeps']) == 0:
                    for s in range(1, S):          # the key frame's slot again (row None), time lag 0, remove_close
                        row.append(None)
                        counts[b, s] = key.shape[0]
                        flags[b, s] = L.SWEEP_TIME_LAG | close
                else:
                    for s, idx in enumerate(choose_sweeps(len(smp['sweeps']), sw['sweeps_num'], sw['test_mode']), 1):
                        sweep = smp['sweeps'][idx]
                        pts = _read_points(sweep['data_path'], sw['load_dim'])
                        self._check_cap(pts, sweep['data_path'])
                        row.append(pts)
                        counts[b, s] = pts.shape[0]
                        flags[b, s] = L.SWEEP_TRANSFORM | L.SWEEP_TIME_LAG | close
                        poses[b, s, :9] = np.asarray(sweep['sensor2lidar_rotation'], np.float64).reshape(9)
                        poses[b, s, 9:] = np.asarray(sweep['sensor2lidar_translation'], np.float64).reshape(3)
                        lags[b, s] = ts - sweep['timestamp'] / 1e6
            row += [np.zeros((0, self.width), np.float32)] * (S - len(row))
            files.append(row)
        return files, flags, counts, poses, lags

    def _check_cap(self, pts, src):
        if pts.shape[0] > self.max_points:
            name = src if isinstance(src, (str, os.PathLike)) else 'array'
            raise ValueError(f'{name}: {pts.shape[0]} points exceed the loader capacity max_points={self.max_points}')

    # ------------------------------------------------------------------ device side
    def _alloc(self):
        B, S, dev = self.batch_size, self.n_src, self.device
        self._dev = dict(
            files=torch.empty((B, S, self.max_points, self.width), dtype=torch.float32, device=dev),
            counts=torch.zeros((B, S), dtype=torch.int32, device=dev),
            poses=torch.zeros((B, S, 12), dtype=torch.float64, device=dev),
            lags=torch.zeros((B, S), dtype=torch.float32, device=dev),
            out=torch.empty((B, self.capacity, self.n_cols), dtype=torch.float32, device=dev),
            total=torch.zeros((B,), dtype=torch.int32, device=dev))
        self._host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
                      for k, v in self._dev.items() if k in ('files', 'counts', 'poses', 'lags')}
        self._srcs = []
        lib = L.load()
        ws = 0
        for b in range(B):
            srcs = (L.SweepSrc * S)()
            for s in range(S):
                srcs[s] = L.SweepSrc(self._dev['files'][b, s].data_ptr(), self.max_points, self.width, 0)
            self._srcs.append(srcs)
            ws = max(ws, lib.srf_merge_sweeps_ws_bytes(srcs, S))
        self._ws = torch.empty((B, (ws + 255) // 256 * 256), dtype=torch.uint8, device=dev)
        self._cols = (ctypes.c_int32 * self.n_cols)(*self.cols)
        rng = self.steps.point_cloud_range
        self._range = (ctypes.c_float * 6)(*rng) if rng is not None else None

    def stage(self, samples):
        files, flags, counts, poses, lags = self.read(samples)
        if self._dev is None:
            self._alloc()
        if self._copied is not None:
            self._copied.synchronize()             # the previous stage's copies still read the pinned buffers
        h, d = self._host, self._dev
        stream = torch.cuda.current_stream(self.device)
        for b, row in enumerate(files):
            for s, pts in enumerate(row):
                if pts is None or pts.shape[0] == 0:
                    continue
                n = pts.shape[0]
                h['files'][b, s, :n].numpy()[...] = pts
                d['files'][b, s, :n].copy_(h['files'][b, s, :n], non_blocking=True)
        for k, v in (('counts', counts), ('poses', poses), ('lags', lags)):
            h[k].numpy()[...] = v
            d[k].copy_(h[k], non_blocking=True)
        self._flags = flags
        self._slots = [[0 if s and row[s] is None else s for s in range(self.n_src)] for row in files]
        self._copied = torch.cuda.Event()
        self._copied.record(stream)

    def __call__(self):
        if self._dev is None:
            raise RuntimeError('stage() samples before running the loader')
        d, lib, S = self._dev, L.load(), self.n_src
        for b in range(self.batch_size):
            srcs = self._srcs[b]
            for s in range(S):
                srcs[s].points = d['files'][b, self._slots[b][s]].data_ptr()
                srcs[s].flags = int(self._flags[b, s])
            L.check(lib.srf_merge_sweeps(srcs, S, d['counts'][b].data_ptr(), d['poses'][b].data_ptr(),
                                         d['lags'][b].data_ptr(), self._cols, self.n_cols, self._range, 1.0,
                                         d['out'][b].data_ptr(), d['total'][b:b + 1].data_ptr(), self._ws[b].data_ptr(),
                                         self._ws.shape[1], L.stream_ptr()), 'srf_merge_sweeps')
        return [d['out'][b] for b in range(self.batch_size)], d['total']


def augment_points(points, views, point_cloud_range=None, count=None):
    """srf_augment_points: one (cap, C) float32 CUDA cloud (first `count` rows valid, a (1,) int32 device tensor; None:
    all) -> (views (A, cap, C), counts (A,) int32 device).  View a = views[a] = (scale, horizontal, vertical): xyz scaled
    in float32, y negated (horizontal), x negated (vertical), then the strict point_cloud_range test when given; kept
    rows first in row order, NaN rows after.  No host synchronisation."""
    pts = points.float().contiguous()
    cap, c = pts.shape
    n = len(views)
    lib = L.load()
    scales = (ctypes.c_float * n)(*[float(s) for s, _, _ in views])
    flips = (ctypes.c_int32 * n)(*[(L.AUG_FLIP_HORIZONTAL if h else 0) | (L.AUG_FLIP_VERTICAL if v else 0) for _, h, v in views])
    need = ctypes.c_size_t(0)
    L.check(lib.srf_augment_points(None, cap, c, None, n, scales, flips, None, None, None, None, ctypes.byref(need), None),
            'srf_augment_points')
    ws = torch.empty(max(int(need.value), 1), dtype=torch.uint8, device=pts.device)
    out = torch.empty((n, cap, c), dtype=torch.float32, device=pts.device)
    counts = torch.empty((n,), dtype=torch.int32, device=pts.device)
    rng = L.f6(point_cloud_range) if point_cloud_range is not None else None
    L.check(lib.srf_augment_points(L.ptr(pts), cap, c, L.ptr(count), n, scales, flips, rng, L.ptr(out), L.ptr(counts),
                                   L.ptr(ws), ctypes.byref(ctypes.c_size_t(ws.numel())), L.stream_ptr()), 'srf_augment_points')
    return out, counts
