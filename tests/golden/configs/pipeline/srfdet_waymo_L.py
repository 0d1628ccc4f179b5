# RESTATEMENT, not a copy of the original file: SRFDet3D's configs/waymo/srfdet_dvoxel_waymo_L.py as far as inference
# from LiDAR files needs it -- the `model` dict of ../model/srfdet_waymo_L.py plus the point steps of `test_pipeline`.
# Assumptions (the original test_pipeline could not be checked; these are the values of mmdet3d 1.0's Waymo LiDAR
# configs): LoadPointsFromFile(load_dim=6, use_dim=5), no sweeps, MultiScaleFlipAug3D(flip=False) around the identity
# GlobalRotScaleTrans, RandomFlip3D and PointsRangeFilter.
import os

exec(open(os.path.join(os.path.dirname(__file__), '..', 'model', 'srfdet_waymo_L.py')).read())

point_cloud_range = [-76.8, -76.8, -2, 76.8, 76.8, 4]
class_names = ['Car', 'Pedestrian', 'Cyclist']
file_client_args = dict(backend='disk')

test_pipeline = [
    dict(type='LoadPointsFromFile', coord_type='LIDAR', load_dim=6, use_dim=5, file_client_args=file_client_args),
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
