"""Host-side logic without a GPU: the reference's configs build the drop-in modules, the
state-dict keys and the layer plan match the reference, frame partition over gloo."""
import json
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle as O

CFGS = {
    'nusc': dict(pts_voxel_layer=dict(max_num_points=10, voxel_size=[0.075, 0.075, 0.2], max_voxels=(120000, 160000),
                                      point_cloud_range=[-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]),
                 pts_voxel_encoder=dict(type='HardSimpleVFE', num_features=5),
                 pts_middle_encoder=dict(type='SparseEncoderCustom', in_channels=5, sparse_shape=[41, 1472, 1472], output_channels=128,
                                         order=('conv', 'norm', 'act'),
                                         encoder_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128)),
                                         encoder_paddings=((0, 0, 1), (0, 0, 1), (0, 0, [0, 1, 1]), (0, 0)), block_type='basicblock')),
    'kitti': dict(pts_voxel_layer=dict(voxel_size=[0.05, 0.05, 0.1], max_num_points=-1, point_cloud_range=[0, -40, -3, 70.4, 40, 1], max_voxels=(-1, -1)),
                  pts_voxel_encoder=dict(type='DynamicVFECustom', in_channels=4, feat_channels=[4], with_distance=False, voxel_size=[0.05, 0.05, 0.1],
                                         with_cluster_center=True, with_voxel_center=True, point_cloud_range=[0, -40, -3, 70.4, 40, 1],
                                         norm_cfg=dict(type='naiveSyncBN1dCustom', eps=1e-3, momentum=0.01)),
                  pts_middle_encoder=dict(type='SparseEncoderCustom', in_channels=4, sparse_shape=[41, 1600, 1408], order=('conv', 'norm', 'act'))),
}


@pytest.fixture(scope='module', autouse=True)
def _built():
    from srfdet_b200 import build
    build.build()


@pytest.mark.parametrize('tag', ['nusc', 'kitti'])
def test_config_builds_drop_in_modules(tag, golden_dir):
    from srfdet_b200.plugin import SRFDetPointPath
    det = SRFDetPointPath(**CFGS[tag], type_unused=None)
    enc = det.pts_middle_encoder
    with open(os.path.join(golden_dir, 'encoder_plan.json')) as f:
        rec = json.load(f)[tag]
    # flat conv list equals what the reference constructor requested from mmdet3d
    flat = []
    for c in rec['calls']:
        if c['fn'] == 'SparseBasicBlock':
            flat += [(True, c['cin'], c['cout']), (True, c['cout'], c['cout'])]
        else:
            flat.append((c['conv_type'] == 'SubMConv3d', c['cin'], c['cout']))
    plan = enc.layer_plan()
    assert [(cv.subm, cv.in_channels, cv.out_channels) for cv, _, _, _ in plan] == flat
    # ... and equals the oracle's independent restatement
    e = CFGS[tag]['pts_middle_encoder']
    oplan = O.encoder_layer_plan(e['in_channels'], 16, e.get('output_channels', 128),
                                 e.get('encoder_channels', ((16,), (32, 32, 32), (64, 64, 64), (64, 64, 64))),
                                 e.get('encoder_paddings', ((1,), (1, 1, 1), (1, 1, 1), ((0, 1, 1), 1, 1))),
                                 e.get('block_type', 'conv_module'))
    for (cv, bn, sv, ad), L in zip(plan, oplan):
        assert cv.kernel_size == tuple(L['ksize']) and cv.stride == tuple(L['stride'])
        if not cv.subm:
            assert cv.padding == tuple(L['pad'])
        assert bool(L.get('save_identity')) == sv and bool(L.get('add_identity')) == ad
    keys = set(enc.state_dict().keys())
    for L in oplan:
        assert f"{L['name']}.{L['conv']}.weight" in keys
        assert f"{L['name']}.{L['bn']}.running_var" in keys
    w = enc.state_dict()['conv_input.0.weight']
    assert tuple(w.shape) == (16, 3, 3, 3, e['in_channels'])          # spconv-2 layout


def test_reference_config_files_load_if_present(golden_dir):
    """Config files in the reference's plain-Python form (tests/golden/configs: the model sections of two of its configs)
    build the modules."""
    from srfdet_b200.plugin import SRFDetPointPath, build_head, build_roi_extractor, load_config
    with open(os.path.join(golden_dir, 'encoder_plan.json')) as f:
        recorded = json.load(f)
    for tag, name in [('waymo', 'waymo/srfdet_dvoxel_waymo_L.py'), ('nusc', 'nus/srfdet_voxel_nusc_LC.py')]:
        enc = dict(load_config(os.path.join(golden_dir, 'configs', name))['model']['pts_middle_encoder'])
        assert enc.pop('type') == 'SparseEncoderCustom'
        assert json.loads(json.dumps(enc)) == recorded[tag]['cfg']        # what the original config files hold
    det = SRFDetPointPath.from_config(os.path.join(golden_dir, 'configs', 'waymo', 'srfdet_dvoxel_waymo_L.py'))
    assert det.is_dynamic and len(det.pts_middle_encoder.layer_plan()) == 21
    cfg = load_config(os.path.join(golden_dir, 'configs', 'nus', 'srfdet_voxel_nusc_LC.py'))['model']['bbox_head']
    head = build_head(cfg['single_head_lidar'] | dict(num_classes=10, feat_channels=128))
    assert head.use_fusion and head.inst_interact_lidar.dynamic_dim == 32
    pooler = build_roi_extractor(cfg['roi_extractor_img'])
    assert pooler.num_inputs == 4 and pooler.featmap_strides == [4, 8, 16, 32]


def test_training_mode_is_rejected():
    from srfdet_b200.plugin import SparseEncoderCustom
    enc = SparseEncoderCustom(in_channels=4, sparse_shape=[41, 1600, 1408]).train()
    with pytest.raises(NotImplementedError):
        enc(torch.zeros(1, 4), torch.zeros(1, 4, dtype=torch.int32), 1)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from srfdet_b200 import frames
    local = frames.run_partitioned(7, lambda i: torch.full((2,), float(i * 10 + rank)))
    assert sorted(local) == list(range(rank, 7, world))
    allr = frames.gather_results(local, 7)
    t = frames.max_over_ranks(1.0 + rank, 'cpu')
    if rank == 0:
        torch.save(dict(vals=[float(x[0]) for x in allr], tmax=t), out)
    dist.barrier()
    dist.destroy_process_group()


def test_frame_partition_gloo_world2(tmp_path):
    """N>1 path: frames round-robin over 2 ranks, no data-path collective, results gathered."""
    out = str(tmp_path / 'r.pt')
    mp.spawn(_worker, args=(2, 29731, out), nprocs=2, join=True)
    r = torch.load(out)
    assert r['vals'] == [0.0, 11.0, 20.0, 31.0, 40.0, 51.0, 60.0]
    assert r['tmax'] == 2.0


def test_spconv1_layout_checkpoint_loads_bit_exact():
    """A state dict in the spconv-1 / mmcv weight layout (kD,kH,kW,Cin,Cout) loads into
    SparseEncoderCustom -- through the PARENT module's load_state_dict -- and yields exactly the
    spconv-2 weights (SURVEY.md 8f rank 4: checkpoint import)."""
    import torch
    from srfdet_b200.plugin import SparseEncoderCustom
    kw = dict(in_channels=5, sparse_shape=[41, 1472, 1472], output_channels=128,
              encoder_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128)),
              encoder_paddings=((0, 0, 1), (0, 0, 1), (0, 0, [0, 1, 1]), (0, 0)), block_type='basicblock')
    torch.manual_seed(0)
    a = SparseEncoderCustom(**kw)
    holder_a = torch.nn.ModuleDict(dict(pts_middle_encoder=a))
    sd1 = {}
    n_conv = 0
    for k, v in holder_a.state_dict().items():
        if v.dim() == 5:
            sd1[k] = v.permute(1, 2, 3, 4, 0).contiguous()      # (Cout,kD,kH,kW,Cin) -> (kD,kH,kW,Cin,Cout)
            n_conv += 1
        else:
            sd1[k] = v.clone()
    assert n_conv == 21
    torch.manual_seed(1)
    b = SparseEncoderCustom(**kw)
    holder_b = torch.nn.ModuleDict(dict(pts_middle_encoder=b))
    missing, unexpected = holder_b.load_state_dict(sd1, strict=True)
    assert not missing and not unexpected
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb), ka
    # and the (kvol, cin, cout) views the kernels pack from are identical
    for (ca, *_), (cb, *_) in zip(a.layer_plan(), b.layer_plan()):
        assert torch.equal(ca.kio(), cb.kio())


def test_weight_caches_follow_parent_load_state_dict():
    """Packed / folded weight caches are keyed on (data_ptr, version) of their source tensors, so a
    checkpoint loaded through ANY ancestor module (which never calls a child's load_state_dict) or an
    in-place update invalidates them."""
    import torch
    from srfdet_b200.plugin import DynamicVFECustom, SparseEncoderCustom
    from srfdet_b200.plugin.head import _cached
    enc = SparseEncoderCustom(in_channels=4, sparse_shape=[41, 1600, 1408])
    v0 = enc._weights_version()
    parent = torch.nn.ModuleDict(dict(enc=enc))
    parent.load_state_dict({k: v.clone() for k, v in parent.state_dict().items()})
    v1 = enc._weights_version()
    assert v0 != v1
    with torch.no_grad():
        enc.conv_input[1].running_var.add_(1.0)
    assert enc._weights_version() != v1
    vfe = DynamicVFECustom(in_channels=4, feat_channels=[4], with_cluster_center=True, with_voxel_center=True,
                           voxel_size=[0.05, 0.05, 0.1], point_cloud_range=[0, -40, -3, 70.4, 40, 1],
                           norm_cfg=dict(type='naiveSyncBN1dCustom', eps=1e-3, momentum=0.01))
    w0 = vfe._weights_version()
    torch.nn.ModuleDict(dict(v=vfe)).load_state_dict({'v.' + k: t.clone() for k, t in vfe.state_dict().items()})
    assert vfe._weights_version() != w0
    lin = torch.nn.Linear(8, 8)
    cache, calls = {}, []
    make = lambda: calls.append(1) or len(calls)
    assert _cached(cache, 'k', (lin.weight,), make) == 1 and _cached(cache, 'k', (lin.weight,), make) == 1
    torch.nn.Sequential(lin).load_state_dict({'0.weight': torch.zeros(8, 8), '0.bias': torch.zeros(8)})
    assert _cached(cache, 'k', (lin.weight,), make) == 2
