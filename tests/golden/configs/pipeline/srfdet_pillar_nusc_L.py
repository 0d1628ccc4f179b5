# RESTATEMENT, not a copy of the original file: SRFDet3D's configs/nus/srfdet_pillar_nusc_L.py as far as inference from
# LiDAR files needs it -- the `model` dict of ../model/srfdet_pillar_nusc_L.py plus the point steps of `test_pipeline`.
# Assumptions (the original test_pipeline could not be checked): the nuScenes test_pipeline of
# ./srfdet_nusc_L.py (LoadPointsFromFile, LoadPointsFromMultiSweeps with 10 sweeps, the identity test-time
# augmentations), with PointsRangeFilter at the pillar range [-51.2, -51.2, -5, 51.2, 51.2, 3].
import os

exec(open(os.path.join(os.path.dirname(__file__), '..', 'model', 'srfdet_pillar_nusc_L.py')).read())

point_cloud_range = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
class_names = ['car', 'truck', 'construction_vehicle', 'bus', 'trailer', 'barrier', 'motorcycle', 'bicycle',
               'pedestrian', 'traffic_cone']
file_client_args = dict(backend='disk')

test_pipeline = [
    dict(type='LoadPointsFromFile', coord_type='LIDAR', load_dim=5, use_dim=5, file_client_args=file_client_args),
    dict(type='LoadPointsFromMultiSweeps', sweeps_num=10, use_dim=[0, 1, 2, 3, 4], file_client_args=file_client_args,
         pad_empty_sweeps=True, remove_close=True),
    dict(type='MultiScaleFlipAug3D',
         img_scale=(1333, 800),
         pts_scale_ratio=1,
         flip=False,
         transforms=[
             dict(type='GlobalRotScaleTrans', rot_range=[0, 0], scale_ratio_range=[1.0, 1.0],
                  translation_std=[0, 0, 0]),
             dict(type='RandomFlip3D'),
             dict(type='PointsRangeFilter', point_cloud_range=point_cloud_range),
             dict(type='DefaultFormatBundle3D', class_names=class_names, with_label=False),
             dict(type='Collect3D', keys=['points'])])]
