"""Run an SRFDet checkpoint on point-cloud files: reference config + trained checkpoint in, 3D boxes out, without mmcv.

    python tools/infer.py CONFIG CHECKPOINT --points a.bin [b.bin ...] [--load-dim 5 --use-dim 0 1 2 3 4]
                          [--img-feats feats.npz --lidar2img l2i.npy] [--precision fp16|fp32] [--trusted] [--out results.npz]
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))

EPILOG = """\
Point files are raw float32 arrays of load-dim values per point (mmdet3d LoadPointsFromFile); use-dim selects the
columns the model reads.  Each file is one cloud, used as it is: multi-sweep aggregation (nuScenes
LoadPointsFromMultiSweeps) and the rest of the data pipeline are not part of this tool, so pass clouds that already
hold what the config's pipeline would have produced.  LiDAR-only configs run all clouds as one batch; camera-fusion
configs take one cloud plus the image-neck outputs (the image backbone and neck are not built here): --img-feats is an
.npz with one (n_cam, C, H, W) or (1, n_cam, C, H, W) float32 array per FPN level, in level order, and --lidar2img an
(n_cam, 4, 4) .npy.  --out writes <i>.boxes_3d, <i>.scores_3d and <i>.labels_3d per sample i.
"""


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0], epilog=EPILOG,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('config', help='reference config file (plain Python with a `model` dict)')
    ap.add_argument('checkpoint', help='checkpoint file (a state dict, or a dict with a "state_dict" entry)')
    ap.add_argument('--points', nargs='+', required=True, help='raw float32 point files')
    ap.add_argument('--load-dim', type=int, default=5, help='float32 values per point in the files (default 5)')
    ap.add_argument('--use-dim', type=int, nargs='+', default=None, help='columns passed to the model (default: all)')
    ap.add_argument('--img-feats', help='.npz of image-neck maps, one array per level (fusion configs)')
    ap.add_argument('--lidar2img', help='.npy (n_cam, 4, 4) LiDAR-to-image projections (fusion configs)')
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
        if len(clouds) != 1:
            sys.exit('camera-fusion configs take one cloud per run')
        z = np.load(a.img_feats)
        img_feats = [torch.as_tensor(z[k]).float().cuda() for k in z.files]
        img_feats = [f.unsqueeze(0) if f.dim() == 4 else f for f in img_feats]
        metas[0]['lidar2img'] = np.load(a.lidar2img)
    results = det.simple_test(clouds, metas, img_feats=img_feats)
    out = {}
    for i, (path, r) in enumerate(zip(a.points, results)):
        b = r['pts_bbox']
        for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
            out[f'{i}.{k}'] = b[k].numpy()
        n = b['scores_3d'].numel()
        top = f', top score {float(b["scores_3d"].max()):.3f}' if n else ''
        print(f'{path}: {clouds[i].shape[0]} points, {n} boxes{top}, labels {np.bincount(b["labels_3d"].numpy()).tolist()}')
    if a.out:
        np.savez(a.out, **out)


if __name__ == '__main__':
    main()
