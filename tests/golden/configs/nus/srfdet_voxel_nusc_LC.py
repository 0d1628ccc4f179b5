# The `model` dict of SRFDet3D's configs/nus/srfdet_voxel_nusc_LC.py (:40-179) up to the head's RoI extractors, in the
# reference's plain-Python config form; the image backbone, the head's training settings, the data pipeline, schedule and
# runtime settings are left out.  pts_middle_encoder is the dict make_golden.py recorded from the original
# configs/nus/srfdet_voxel_nusc_L.py into encoder_plan.json, which the LC config shares.
point_cloud_range = [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]
voxel_size = [0.075, 0.075, 0.2]

model = dict(
    type='SRFDet',
    pts_voxel_layer=dict(
        max_num_points=10,
        voxel_size=voxel_size,
        max_voxels=(120000, 160000),
        point_cloud_range=point_cloud_range),
    pts_voxel_encoder=dict(type='HardSimpleVFE', num_features=5),
    pts_middle_encoder=dict(
        type='SparseEncoderCustom',
        in_channels=5,
        sparse_shape=[41, 1472, 1472],
        output_channels=128,
        order=('conv', 'norm', 'act'),
        encoder_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128)),
        encoder_paddings=((0, 0, 1), (0, 0, 1), (0, 0, [0, 1, 1]), (0, 0)),
        block_type='basicblock'),
    bbox_head=dict(
        type='SRFDetHead',
        use_img=True,
        num_classes=10,
        feat_channels_lidar=128,
        feat_channels_img=256,
        hidden_dim=128,
        num_proposals=900,
        num_heads=5,
        single_head_lidar=dict(
            type='SingleSRFDetHead',
            use_fusion=True,
            num_cls_convs=2,
            num_reg_convs=3,
            dim_feedforward=512,
            num_heads=8,
            dropout=0.1,
            act_cfg=dict(type='ReLU', inplace=True),
            dynamic_conv=dict(dynamic_dim=32, dynamic_num=2),
            pc_range=point_cloud_range,
            voxel_size=voxel_size,
            bbox_weights=[1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 0.2, 0.2]),
        roi_extractor_lidar=dict(
            type='SingleRoIExtractor',
            roi_layer=dict(type='RoIAlign', output_size=7, sampling_ratio=2),
            out_channels=128,
            featmap_strides=[8, 16, 32, 64]),
        roi_extractor_img=dict(
            type='SingleRoIExtractor',
            roi_layer=dict(type='RoIAlign', output_size=7, sampling_ratio=2),
            out_channels=128,
            featmap_strides=[4, 8, 16, 32])))
