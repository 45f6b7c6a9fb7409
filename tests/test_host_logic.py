"""CPU tests of the host-side mirror: registry/config plumbing, state_dict
contract, geometry packing, C-ABI library symbols."""
import ctypes
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import depth_from_motion_b200 as pkg
from depth_from_motion_b200 import capi, modules, registry
from depth_from_motion_b200 import synthetic as syn
from tests.util import DFM_CONFIGS, GOLDEN, STATE_DICT_MODULES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_registry_builds_by_type():
    cfg = dict(type='DfMBackbone', in_channels=32, cv_channels=32, num_hg=1,
               cost_sample_factor=4,
               norm_cfg=dict(type='GN', num_groups=32, requires_grad=True))
    cfg.update(depth_cfg=syn.depth_cfg_for(72))  # detectors/dfm.py:45-48
    m = pkg.build_backbone(cfg)
    assert isinstance(m, modules.DfMBackbone) and m.num_planes == 72
    assert m.aggregate_cost.weight.shape == (72, 144, 1, 1)
    n = pkg.build_neck(dict(type='DfMNeck', in_channels=64, out_channels=256,
                            num_frames=2))
    assert isinstance(n, modules.DfMNeck)
    with pytest.raises(KeyError):
        pkg.build_backbone(dict(type='NoSuchBackbone'))


# reference state_dict contract (SURVEY.md section 8a "State")
EXPECTED_KEYS = {
    'dres0.conv.weight': (32, 64, 3, 3, 3), 'dres0.gn.weight': (32,),
    'hg_stereo.0.conv1.0.0.weight': (64, 32, 3, 3, 3),
    'hg_stereo.0.conv1.0.1.bias': (64,),
    'hg_stereo.0.conv2.0.weight': (64, 64, 3, 3, 3),
    'hg_stereo.0.conv5.0.weight': (64, 64, 3, 3, 3),
    'hg_stereo.0.conv6.0.weight': (64, 32, 3, 3, 3),
    'pred_stereo.0.0.conv.weight': (32, 32, 3, 3, 3),
    'pred_stereo.0.1.weight': (1, 32, 3, 3, 3),
    'dres0_mono.conv.weight': (32, 32, 3, 3, 3),
    'hg_mono.0.conv4.0.1.weight': (64,),
    'pred_mono.0.1.weight': (1, 32, 3, 3, 3),
    'aggregate_cost.weight': (72, 144, 1, 1),
}


def test_state_dict_contract():
    m = modules.DfMBackbone(in_channels=32, depth_cfg=syn.depth_cfg_for(72))
    sd = m.state_dict()
    assert len(sd) == 57
    assert sum(v.numel() for v in sd.values()) == 1313344  # SURVEY 8a
    for k, shp in EXPECTED_KEYS.items():
        assert tuple(sd[k].shape) == shp, k
    params = syn.make_backbone_params(np.random.RandomState(0), 72)
    m.load_state_dict(params, strict=True)
    n = modules.DfMNeck(64, 256, num_frames=2)
    assert sum(v.numel() for k, v in n.state_dict().items()
               if 'running' not in k and 'tracked' not in k) == 15932160
    assert 'mono_layers.0.conv0.conv.weight' in n.state_dict()
    assert 'stereo_layers.5.bn.running_var' in n.state_dict()
    assert 'model.1.conv.weight' in modules.OutdoorImVoxelNeck(64, 256).state_dict()
    f = modules.FrustumToVoxel().state_dict()
    assert {k: tuple(v.shape) for k, v in f.items()} == {
        'voxel_convs.0.0.conv.weight': (32, 64, 3, 3, 3),
        'voxel_convs.0.0.gn.weight': (32,), 'voxel_convs.0.0.gn.bias': (32,)}


def test_state_dict_matches_reference_modules():
    """Key order and shapes equal those of the reference modules' state_dicts
    (tests/golden/state_dict_layout.json)."""
    with open(os.path.join(GOLDEN, 'state_dict_layout.json')) as f:
        gold = json.load(f)
    assert sorted(gold) == sorted(STATE_DICT_MODULES)
    for name, make in STATE_DICT_MODULES.items():
        sd = make(modules).state_dict()
        assert [[k, list(v.shape)] for k, v in sd.items()] == gold[name], name


@pytest.mark.parametrize('cfg_name', DFM_CONFIGS)
def test_reference_configs_parse_and_build_hot_path(cfg_name, tmp_path):
    """The hot-path blocks of configs/dfm/*.py, as the reference parses them
    (tests/golden/config_model_blocks.json), load from a flat config file and build the
    hot-path modules by type."""
    with open(os.path.join(GOLDEN, 'config_model_blocks.json')) as f:
        blocks = json.load(f)[cfg_name]
    path = tmp_path / cfg_name
    path.write_text(f'model = {blocks!r}\n')
    cfg = registry.Config.fromfile(str(path))
    model = cfg.model
    if model['type'] == 'DfM':
        bs = dict(model['backbone_stereo'])
        bs.update(depth_cfg=model['depth_cfg'])
        m = pkg.build_backbone(bs)
        assert m.num_planes == 72
        h = pkg.build_head(dict(model['depth_head']))
        assert isinstance(h, modules.DepthHead) and not h.with_convs
        ft = pkg.build_neck(dict(model['feature_transformation']))
        assert isinstance(ft, modules.FrustumToVoxel) and ft.sem_atten_feat
        vc = model['voxel_cfg']
        nvox = [round((vc['point_cloud_range'][3 + a] - vc['point_cloud_range'][a]) /
                      vc['voxel_size'][a]) for a in range(3)]
        assert nvox == [288, 304, 20]
        b3 = pkg.build_backbone(dict(model['backbone_3d']))       # BEVHourglass, GN variant
        assert isinstance(b3, modules.BEVHourglass) and b3.in_channels == 160
        hd = pkg.build_head(dict(model['bbox_head_3d']))
        assert isinstance(hd, modules.LIGAAnchor3DHead)
        assert (hd.num_anchors, hd.cls_out_channels) == (6, 18)
    else:
        n = pkg.build_neck(dict(model['neck_3d']))
        assert isinstance(n, (modules.DfMNeck, modules.OutdoorImVoxelNeck))


def test_geometry_packing():
    meta = syn.make_img_meta(384, 1248, flip=True, crop_offset=(3, 7), scale=1.25,
                             ori_shape=(370, 1224, 3))
    g = modules.geometry_from_meta(meta)
    assert g.flip == 1 and g.org_w == 1224 and g.scale == 1.25
    assert (g.crop_x, g.crop_y) == (3.0, 7.0)
    assert abs(g.cam2img[0] - 721.5377) < 1e-3 and g.cam2img[15] == 1.0
    assert abs(g.cur2prev[11] - 0.958234025) < 1e-6


def test_no_cpu_fallback():
    m = modules.DfMBackbone(in_channels=32, depth_cfg=syn.depth_cfg_for(8))
    x = torch.zeros(1, 32, 32, 64)
    with pytest.raises(RuntimeError):
        m(x, x, [syn.make_img_meta(32, 64)])


def _header_symbols():
    txt = open(os.path.join(ROOT, 'include', 'dfm_b200.h')).read()
    txt = re.sub(r'/\*.*?\*/', '', txt, flags=re.S)
    return sorted(set(re.findall(r'\b(dfm_[a-z0-9_]+)\s*\(', txt)))


def test_header_and_binding_agree():
    assert _header_symbols() == sorted(capi.SYMBOLS)


@pytest.mark.skipif(shutil.which('nvcc') is None and not capi.library_built(),
                    reason='library not built and no nvcc')
def test_library_exports_every_declared_symbol():
    if not capi.library_built():
        from depth_from_motion_b200 import build
        build.build()
    L = ctypes.CDLL(capi.LIB_PATH)  # dlopen only: no compute call without a GPU
    for s in _header_symbols():
        assert hasattr(L, s), s
    assert L.dfm_version() >= 100
    out = subprocess.run(['cuobjdump', '-lelf', capi.LIB_PATH], capture_output=True,
                         text=True).stdout if shutil.which('cuobjdump') else 'sm_100a'
    assert 'sm_100a' in out


@pytest.mark.skipif(shutil.which('gcc') is None, reason='no C compiler')
def test_ctypes_structs_match_the_c_header(tmp_path):
    """The header is plain C: compile it with gcc and compare sizeof / offsetof of every
    descriptor struct with the ctypes mirror in capi.py (an ABI drift would corrupt
    arguments silently)."""
    structs = {'dfm_geometry_t': capi.Geometry, 'dfm_backbone_desc_t': capi.BackboneDesc,
               'dfm_lift_desc_t': capi.LiftDesc, 'dfm_neck_desc_t': capi.NeckDesc,
               'dfm_frustum_desc_t': capi.FrustumDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>',
             f'#include "{os.path.join(ROOT, "include", "dfm_b200.h")}"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['return 0;', '}']
    src = tmp_path / 'abi.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'abi'
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-o', str(exe), str(src)],
                   check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True,
                                                 check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f'{cname}.{fname}']) == getattr(cls, fname).offset, (cname, fname)


def test_frustum_host_side_contract():
    """FrustumToVoxel mirror: voxel-grid axes are recovered from the injected coordinates_3d
    (detectors/dfm.py:193-211), a non-meshgrid tensor is refused, CPU tensors are refused."""
    c3d = syn.frustum_coordinates(syn.KITTI_POINT_CLOUD_RANGE, (288, 304, 20))
    xs, ys, zs = modules.FrustumToVoxel._separable_centres(c3d)
    assert (len(xs), len(ys), len(zs)) == (288, 304, 20)
    assert abs(float(xs[0]) - 2.1) < 1e-6 and abs(float(ys[-1]) - 30.3) < 1e-5
    assert abs(float(zs[0]) + 2.9) < 1e-6
    bad = c3d.clone()
    bad[3, 5, 7, 0] += 0.01
    with pytest.raises(RuntimeError):
        modules.FrustumToVoxel._separable_centres(bad)
    m = modules.FrustumToVoxel()
    m.coordinates_3d, m.depth_cfg = c3d, syn.depth_cfg_for(8)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 32, 8, 8, 16), modules.CostLogits(torch.zeros(1, 1, 8, 8, 16)),
          [dict(cam2img=np.eye(4).tolist(), pad_shape=(32, 64, 3))], torch.zeros(1, 32, 8, 16))


def test_checkpoint_key_plumbing():
    """A detector-style checkpoint (mmdet3d names, or LIGA-DfM names as handled by the
    reference's tools/model_converters/convert_dfm_checkpoints.py:34-81) is split into the
    hot-path modules and loads with strict=True."""
    from depth_from_motion_b200 import checkpoint as ck
    cfg = syn.depth_cfg_for(8)
    rng = np.random.RandomState(5)
    bb_sd = syn.make_backbone_params(rng, 8)
    ft_sd = syn.make_frustum_case(7, 32, 64, 8, (8, 8, 4))['params']
    det = {}
    for k, v in bb_sd.items():
        det['backbone_stereo.' + k] = v
    for k, v in ft_sd.items():
        det['feature_transformation.' + k] = v
    det['backbone.layer1.0.conv1.weight'] = torch.zeros(3)
    det['bbox_head_3d.conv_cls.weight'] = torch.zeros(3)
    bb = modules.DfMBackbone(in_channels=32, depth_cfg=cfg)
    ft = modules.FrustumToVoxel()
    ck.load_hot_path({'state_dict': det}, backbone=bb, frustum=ft)
    assert all(torch.equal(bb.state_dict()[k], v) for k, v in bb_sd.items())
    assert all(torch.equal(ft.state_dict()[k], v) for k, v in ft_sd.items())
    # LIGA-DfM names: backbone_3d.* is the stereo backbone except its image backbone / necks
    # and the voxel convs
    liga = {'global_step': torch.zeros(1)}
    for k, v in bb_sd.items():
        liga['backbone_3d.' + k] = v
    for k, v in ft_sd.items():
        liga['backbone_3d.rpn3d_convs.' + k[len('voxel_convs.'):]] = v
    liga['backbone_3d.feature_backbone.conv1.weight'] = torch.zeros(3)
    liga['lidar_model.backbone_3d.conv1.0.weight'] = torch.zeros(3)
    assert ck.convert_liga_key('backbone_3d.feature_neck.x') == 'neck.x'
    assert ck.convert_liga_key('backbone_3d.dres0.conv.weight') == \
        'backbone_stereo.dres0.conv.weight'
    assert ck.convert_liga_key('lidar_model.backbone_3d.conv1.0.weight').startswith('lidar_model')
    bb2 = modules.DfMBackbone(in_channels=32, depth_cfg=cfg)
    ft2 = modules.FrustumToVoxel()
    ck.load_hot_path({'model_state': liga}, backbone=bb2, frustum=ft2)
    assert all(torch.equal(bb2.state_dict()[k], v) for k, v in bb_sd.items())
    assert all(torch.equal(ft2.state_dict()[k], v) for k, v in ft_sd.items())
    with pytest.raises(KeyError):
        ck.load_hot_path({'state_dict': {'x.y': torch.zeros(1)}}, backbone=bb2)


def test_param_sync_hooks_and_guards():
    """ADVICE r1: `_version` does not see writes through `.data`; load_state_dict / train() /
    eval() and mark_dirty() must force a re-upload; unsupported configs fail loudly."""
    m = modules.DfMBackbone(in_channels=32, depth_cfg=syn.depth_cfg_for(8))
    uploads = []
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    n0 = len(uploads)
    assert n0 == 57
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    assert len(uploads) == n0                      # unchanged -> no upload
    m.dres0.conv.weight.data.fill_(1.0)            # invisible to (data_ptr, _version) ...
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    assert len(uploads) == n0
    m.sync_params()                                # ... hence the explicit call
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    assert len(uploads) == 2 * n0
    m.load_state_dict(m.state_dict())
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    assert len(uploads) == 3 * n0
    m.eval()
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    assert len(uploads) == 4 * n0
    with torch.no_grad():
        m.dres1.gn.bias.add_(1.0)                  # bumps _version
    m._sync.sync(m, lambda k, p, n: uploads.append(k))
    assert len(uploads) == 5 * n0
    # content fingerprint (DFM_PARAM_CHECK=1 path)
    f0 = modules._ParamSync.fingerprint(m)
    m.dres0.conv.weight.data.mul_(0.5)
    assert not torch.equal(f0, modules._ParamSync.fingerprint(m))
    # forward-only guard in training mode
    m.train()
    with pytest.raises(RuntimeError, match='forward-only'):
        m._forward_only(torch.zeros(1))
    with torch.no_grad():
        m._forward_only(torch.zeros(1))
    m.eval()
    m._forward_only(torch.zeros(1))
    with pytest.raises(AssertionError):
        modules.DfMBackbone(in_channels=32, depth_cfg=syn.depth_cfg_for(8),
                            norm_cfg=dict(type='GN', num_groups=16))
    meta = dict(pcd_rotation=np.eye(3), pcd_scale_factor=1.0)
    modules._require_identity_3d_aug(meta)
    with pytest.raises(NotImplementedError):
        modules._require_identity_3d_aug(dict(pcd_scale_factor=1.05))
    with pytest.raises(NotImplementedError):
        modules._require_identity_3d_aug(dict(pcd_horizontal_flip=True))


def test_bev_stage_state_dict_contract():
    """BEVHourglass / LIGAAnchor3DHead mirrors take the reference state_dict keys (the same
    dicts load strict=True into the verbatim reference classes in tests/golden/make_golden.py)
    and build from the KITTI config block through the registry."""
    gn = dict(type='GN', num_groups=32, requires_grad=True)
    c = syn.make_bev_case(seed=1, nz=5, ny=8, nx=8)
    bev = pkg.build_backbone(dict(type='BEVHourglass', in_channels=160, out_channels=64,
                                  norm_cfg=gn))
    bev.load_state_dict(c['bev'], strict=True)
    head = registry.HEADS.build(dict(
        type='LIGAAnchor3DHead', num_classes=3, in_channels=64, feat_channels=64, num_convs=2,
        use_direction_classifier=True, diff_rad_by_sin=True, dir_offset=0.7854,
        anchor_generator=dict(type='Anchor3DRangeGenerator',
                              ranges=[[2, -30.4, -1.78, 59.6, 30.4, -1.78]] * 3,
                              sizes=[[3.9, 1.6, 1.56], [0.8, 0.6, 1.73], [1.76, 0.6, 1.73]],
                              rotations=[0, 1.57], reshape_out=False),
        assign_per_class=True, bbox_coder=dict(type='DeltaXYZWLHRBBoxCoder'),
        loss_cls=dict(type='FocalLoss'), loss_bbox=dict(type='SmoothL1Loss'),
        loss_dir=dict(type='CrossEntropyLoss'), loss_iou=dict(type='IOU3DLoss'), norm_cfg=gn))
    head.load_state_dict(c['head'], strict=True)
    assert head.num_anchors == 6 and head.box_code_size == 7
    assert head.conv_cls.out_channels == 18 and head.conv_reg.out_channels == 42
    assert head.conv_dir_cls.out_channels == 12
    with pytest.raises(AssertionError):   # the SyncBN (LiDAR teacher) variant is not mirrored
        modules.BEVHourglass(160, 64, norm_cfg=dict(type='SyncBN'))
    with pytest.raises(RuntimeError):     # no CPU path
        bev(torch.zeros(1, 160, 8, 8))
