# The point-cloud part of the `model` dict of SRFDet3D's configs/waymo/srfdet_dvoxel_waymo_L.py (:6-10, :26-59), in the
# reference's plain-Python config form; the head, data pipeline, schedule and runtime settings are left out.
# pts_middle_encoder is the dict make_golden.py recorded from the original file into encoder_plan.json.
point_cloud_range = [-76.8, -76.8, -2, 76.8, 76.8, 4]
voxel_size = [0.1, 0.1, 0.15]

model = dict(
    type='SRFDetWaymo',
    pts_voxel_layer=dict(
        voxel_size=voxel_size,
        max_num_points=-1,
        point_cloud_range=point_cloud_range,
        max_voxels=(-1, -1)),
    pts_voxel_encoder=dict(
        type='DynamicVFECustom',
        in_channels=5,
        feat_channels=[5, 5],
        with_distance=False,
        voxel_size=voxel_size,
        with_cluster_center=True,
        with_voxel_center=True,
        point_cloud_range=point_cloud_range,
        norm_cfg=dict(type='naiveSyncBN1dCustom', eps=1e-3, momentum=0.01)),
    pts_middle_encoder=dict(
        type='SparseEncoderCustom',
        in_channels=5,
        sparse_shape=[41, 1536, 1536],
        output_channels=128,
        order=('conv', 'norm', 'act'),
        encoder_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128)),
        encoder_paddings=((0, 0, 1), (0, 0, 1), (0, 0, [0, 1, 1]), (0, 0)),
        block_type='basicblock'))
