# RESTATEMENT, not a copy of an original file: ../pipeline/srfdet_nusc_L.py with flip test-time augmentation, the
# "double flip" setting of mmdet3d's nuScenes LiDAR configs: MultiScaleFlipAug3D(flip=True, pcd_horizontal_flip=True,
# pcd_vertical_flip=True) around RandomFlip3D(sync_2d=False), 8 views of which 4 are distinct.
# Assumptions (no original SRFDet TTA config could be checked):
#   - the point steps, the identity GlobalRotScaleTrans and the PointsRangeFilter inside the wrapper are those of
#     ../pipeline/srfdet_nusc_L.py
#   - test_cfg.pts.max_num = 500 (merge_aug_bboxes_3d reads it; none of the shipped configs sets it)
import os

exec(open(os.path.join(os.path.dirname(__file__), 'srfdet_nusc_L.py')).read())

model['test_cfg']['pts']['max_num'] = 500

test_pipeline = [
    dict(type='LoadPointsFromFile', coord_type='LIDAR', load_dim=5, use_dim=5, file_client_args=file_client_args),
    dict(type='LoadPointsFromMultiSweeps', sweeps_num=10, use_dim=[0, 1, 2, 3, 4], file_client_args=file_client_args,
         pad_empty_sweeps=True, remove_close=True),
    dict(type='MultiScaleFlipAug3D',
         img_scale=(1333, 800),
         pts_scale_ratio=1,
         flip=True,
         pcd_horizontal_flip=True,
         pcd_vertical_flip=True,
         transforms=[
             dict(type='GlobalRotScaleTrans', rot_range=[0, 0], scale_ratio_range=[1.0, 1.0],
                  translation_std=[0, 0, 0]),
             dict(type='RandomFlip3D', sync_2d=False),
             dict(type='PointsRangeFilter', point_cloud_range=point_cloud_range),
             dict(type='DefaultFormatBundle3D', class_names=class_names, with_label=False),
             dict(type='Collect3D', keys=['points'])])]
