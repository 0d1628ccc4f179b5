# RESTATEMENT, not a copy of the original file: SRFDet3D's configs/nus/srfdet_voxel_nusc_L.py as far as inference from
# LiDAR files needs it -- the `model` dict of ../model/srfdet_nusc_L.py plus the point steps of `test_pipeline`.
# Assumptions (the original test_pipeline could not be checked; these are the values of the nuScenes LiDAR configs of
# the mmdet3d 1.0 generation this project derives from):
#   - LoadPointsFromFile(load_dim=5, use_dim=5)
#   - LoadPointsFromMultiSweeps(sweeps_num=10, use_dim=[0, 1, 2, 3, 4], pad_empty_sweeps=True, remove_close=True);
#     test_mode is left at its default (False)
#   - MultiScaleFlipAug3D(flip=False) around the identity GlobalRotScaleTrans, RandomFlip3D and PointsRangeFilter
import os

exec(open(os.path.join(os.path.dirname(__file__), '..', 'model', 'srfdet_nusc_L.py')).read())

point_cloud_range = [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]
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
