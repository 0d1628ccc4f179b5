"""Run an SRFDet checkpoint on point-cloud files: reference config + trained checkpoint in, 3D boxes out, without mmcv.

    python tools/infer.py CONFIG CHECKPOINT --points a.bin [b.bin ...] [--load-dim 5 --use-dim 0 1 2 3 4]
                          [--img-feats feats.npz --lidar2img l2i.npy] [--precision fp16|fp32] [--trusted] [--out results.npz]
    python tools/infer.py CONFIG CHECKPOINT --info nuscenes_infos_val.pkl --index 0 1 2 [--data-root data/nuscenes]
                          [--max-points 40000] [--precision fp16|fp32] [--trusted] [--out results.npz]
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))

EPILOG = """\
--points: point files are raw float32 arrays of load-dim values per point (mmdet3d LoadPointsFromFile); use-dim selects
the columns the model reads.  Each file is one cloud, used as it is, so pass clouds that already hold what the config's
pipeline would have produced.  All clouds run as one batch.  Camera-fusion configs also take the image-neck outputs
(the image backbone and neck are not built here): --img-feats is an .npz with one float32 array per FPN level, in level
order, each (B, n_cam, C, H, W) with one sample per --points file in the same order (or (n_cam, C, H, W) for one cloud),
and --lidar2img a (B, n_cam, 4, 4) .npy (or (n_cam, 4, 4) for one cloud).  Sample i is fused with its own maps and
projections only, as B separate runs of one cloud would be.
--info: frames --index of an mmdet3d nuscenes_infos_*.pkl (read without running any pickled code) go through the point
steps of the config's test_pipeline on the GPU -- LoadPointsFromFile, LoadPointsFromMultiSweeps (the key frame and its
sweeps moved into the key frame's LiDAR frame, with the time lag column) and PointsRangeFilter -- one frame at a time
into a fixed-capacity cloud, so one CUDA graph serves every frame.  --data-root re-roots the infos' paths at their
samples/ or sweeps/ component; --max-points is the capacity per point file (a larger file is an error).  LiDAR-only
configs.  The image pipeline is not part of this tool.
Test-time augmentation: when the config's test_pipeline augments (MultiScaleFlipAug3D with flip=True or scale ratios
other than 1), --info and --points run SRFDet.infer_aug with its distinct views -- the clouds flipped and scaled on the
GPU, all views as one batch, the views' boxes mapped back and merged by class-wise rotated BEV NMS
(merge_aug_bboxes_3d, test_cfg.max_num boxes) -- one CUDA graph for the whole --info sequence.  LiDAR-only configs.
--out writes <i>.boxes_3d, <i>.scores_3d and <i>.labels_3d per sample i.
"""


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0], epilog=EPILOG,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('config', help='reference config file (plain Python with a `model` dict)')
    ap.add_argument('checkpoint', help='checkpoint file (a state dict, or a dict with a "state_dict" entry)')
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument('--points', nargs='+', help='raw float32 point files')
    src.add_argument('--info', help="mmdet3d nuscenes_infos_*.pkl: run the config's point pipeline on frames --index")
    ap.add_argument('--index', type=int, nargs='+', default=[0], help='--info: frame indices (default 0)')
    ap.add_argument('--data-root', help='--info: directory the infos\' samples/ and sweeps/ paths are re-rooted at')
    ap.add_argument('--max-points', type=int, default=40000, help='--info: capacity per point file (default 40000)')
    ap.add_argument('--load-dim', type=int, default=5, help='float32 values per point in the files (default 5)')
    ap.add_argument('--use-dim', type=int, nargs='+', default=None, help='columns passed to the model (default: all)')
    ap.add_argument('--img-feats', help='.npz of image-neck maps, one array per level (fusion configs)')
    ap.add_argument('--lidar2img', help='.npy (B, n_cam, 4, 4) LiDAR-to-image projections, one set per cloud (fusion configs)')
    ap.add_argument('--precision', choices=['fp16', 'fp32'], default=None, help='default: the library default (fp16)')
    ap.add_argument('--trusted', action='store_true',
                    help='allow pickled Python objects in the checkpoint (mmcv checkpoints carry them); only for trusted files')
    ap.add_argument('--out', help='write the results to this .npz')
    a = ap.parse_args(argv)

    import torch
    from srfdet_b200.plugin import SRFDet, set_precision
    if not torch.cuda.is_available():
        sys.exit('tools/infer.py needs a CUDA device (there is no CPU fallback)')
    if a.precision:
        set_precision(a.precision)
    det = SRFDet.from_config(a.config).cuda()
    keys = det.load_checkpoint(a.checkpoint, strict=True, trusted=a.trusted)
    if keys.set_aside_keys:
        print(f'checkpoint: {len(keys.set_aside_keys)} image backbone / neck entries set aside (modules not built)')
    if a.info:
        return run_infos(det, a)
    use_dim = a.use_dim if a.use_dim is not None else list(range(a.load_dim))
    clouds = []
    for path in a.points:
        raw = np.fromfile(path, dtype=np.float32)
        if raw.size % a.load_dim:
            sys.exit(f'{path}: {raw.size} float32 values are not a multiple of --load-dim {a.load_dim}')
        clouds.append(torch.as_tensor(np.ascontiguousarray(raw.reshape(-1, a.load_dim)[:, use_dim])).cuda())
    img_feats, metas = None, [{} for _ in clouds]
    if det.bbox_head.use_img:
        if not (a.img_feats and a.lidar2img):
            sys.exit('this is a camera-fusion config: pass --img-feats and --lidar2img')
        maps, l2i = camera_inputs(np.load(a.img_feats), np.load(a.lidar2img), len(clouds))
        img_feats = [torch.as_tensor(f).float().cuda() for f in maps]
        for m, p in zip(metas, l2i):
            m['lidar2img'] = p
    aug = test_augmentation(a.config)
    if aug is not None:
        results = aug_results(det, det.infer_aug(clouds, aug.views, aug.view_range))
    else:
        results = det.simple_test(clouds, metas, img_feats=img_feats)
    out = {}
    for i, (path, r) in enumerate(zip(a.points, results)):
        report(out, i, path, clouds[i].shape[0], r)
    if a.out:
        np.savez(a.out, **out)


def camera_inputs(z, lidar2img, n_clouds):
    """--img-feats levels and --lidar2img for n_clouds samples -> ((B, n_cam, C, H, W) arrays, (B, n_cam, 4, 4)); exits
    with a message when the counts do not match."""
    maps = [np.asarray(z[k]) for k in z.files]
    if not maps:
        sys.exit('--img-feats holds no arrays')
    if any(f.ndim not in (4, 5) for f in maps):
        sys.exit(f'--img-feats: each level must be (B, n_cam, C, H, W) or (n_cam, C, H, W), got {[f.shape for f in maps]}')
    maps = [f[None] if f.ndim == 4 else f for f in maps]
    if any(f.shape[:2] != maps[0].shape[:2] for f in maps):
        sys.exit(f'--img-feats: every level needs the same (B, n_cam), got {[f.shape[:2] for f in maps]}')
    b, n_cam = maps[0].shape[:2]
    if b != n_clouds:
        sys.exit(f'--img-feats holds maps of {b} sample(s) for {n_clouds} --points file(s): pass one sample per cloud')
    lidar2img = np.asarray(lidar2img, np.float32)
    shape = lidar2img.shape
    if shape == (n_cam, 4, 4) and n_clouds == 1:
        lidar2img = lidar2img[None]
    elif shape != (n_clouds, n_cam, 4, 4):
        sys.exit(f'--lidar2img {shape} does not match {n_clouds} cloud(s) of {n_cam} cameras: pass ({n_clouds}, {n_cam}, 4, 4)')
    return maps, lidar2img


def report(out, i, name, n_points, r):
    b = r['pts_bbox']
    for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
        out[f'{i}.{k}'] = b[k].numpy()
    n = b['scores_3d'].numel()
    top = f', top score {float(b["scores_3d"].max()):.3f}' if n else ''
    print(f'{name}: {n_points} points, {n} boxes{top}, labels {np.bincount(b["labels_3d"].numpy()).tolist()}')


def test_augmentation(config):
    """PointAugmentation of the config's test_pipeline when it augments (flip=True or scale ratios other than 1), else
    None."""
    from srfdet_b200.plugin import registry
    from srfdet_b200.plugin.points import parse_test_augmentations
    cfg = registry.load_config(config)

    def augments(steps):
        for st in steps:
            if st.get('type') == 'MultiScaleFlipAug3D':
                r = st.get('pts_scale_ratio', 1)
                if st.get('flip', False) or (list(r) if isinstance(r, (list, tuple)) else [r]) != [1]:
                    return True
        return False
    if not augments(cfg.get('test_pipeline') or []):
        return None
    return parse_test_augmentations(cfg['test_pipeline'])


def aug_results(det, out):
    """infer_aug outputs -> simple_test-style results (one read-back)."""
    return [dict(pts_bbox=dict(boxes_3d=bx.cpu(), scores_3d=sc.cpu(), labels_3d=lb.cpu())) for bx, sc, lb in det.bbox_head.format_nms(*out)]


def run_infos(det, a):
    from srfdet_b200.plugin import registry
    from srfdet_b200.plugin.points import MultiSweepLoader, load_nuscenes_infos
    cfg = registry.load_config(a.config)
    if 'test_pipeline' not in cfg:
        sys.exit(f'{a.config} has no test_pipeline: --info runs the point steps of the config\'s test_pipeline '
                 '(use --points for clouds that are already merged)')
    if det.bbox_head.use_img:
        sys.exit('--info runs LiDAR-only configs (the image pipeline is not part of this tool)')
    infos = load_nuscenes_infos(a.info, data_root=a.data_root)
    aug = test_augmentation(a.config)
    if aug is not None:
        loader = MultiSweepLoader(aug.loader_steps, batch_size=1, max_points=a.max_points)
    else:
        loader = MultiSweepLoader.from_config(cfg, batch_size=1, max_points=a.max_points)
    det.use_graph = True
    out = {}
    for i, idx in enumerate(a.index):
        if not 0 <= idx < len(infos):
            sys.exit(f'--index {idx}: {a.info} has {len(infos)} frames')
        loader.stage([infos[idx]])
        clouds, counts = loader()
        if aug is not None:
            results = aug_results(det, det.infer_aug(clouds, aug.views, aug.view_range, counts=counts))
        else:
            results = det.simple_test(clouds, [{}])
        report(out, i, infos[idx]['lidar_path'], int(counts[0]), results[0])
    if a.out:
        np.savez(a.out, **out)


if __name__ == '__main__':
    main()
