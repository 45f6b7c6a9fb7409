"""Generates the golden fixtures in this directory from the UNMODIFIED reference
sources (executed verbatim through oracle/ref_loader.py).  Runs only in the build
container, where /root/reference is mounted:

    python tests/golden/make_golden.py

Inputs are regenerated from fixed NumPy seeds by depth_from_motion_b200.synthetic
(and stored too, so a fixture is self-contained); outputs are what the
reference's own DfMBackbone / DepthHead / DfMNeck / OutdoorImVoxelNeck /
FrustumToVoxel / point_sample code returns on CPU in fp32.
"""
import copy
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from depth_from_motion_b200 import synthetic as syn  # noqa: E402
from oracle import dfm_oracle as O  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

KITTI_CASES = {
    # name: (seed, H, W, D, flip, crop, scale, ori_shape)
    'kitti_plain': (11, 32, 64, 8, False, (0, 0), 1.0, None),
    'kitti_aug': (12, 32, 64, 8, True, (10, 40), 1.03, (375, 1242, 3)),
}


def kitti_case(ns, name, spec):
    seed, h, w, d, flip, crop, scale, ori = spec
    cur, prev, metas, params = syn.make_kitti_pair(
        seed, h, w, d, flip=flip, crop_offset=crop, scale=scale, ori_shape=ori)
    cfg = syn.depth_cfg_for(d)
    m = ns.DfMBackbone(in_channels=32, depth_cfg=cfg).eval()
    m.load_state_dict(params, strict=True)
    m.downsampled_depth = O.downsampled_depth(cfg)
    head = ns.DepthHead(
        depth_cfg=dict(mode='UD', num_bins=cfg['num_bins'], min_depth=2,
                       max_depth=59.6), with_convs=False, num_views=1,
        depth_loss=dict(type='balanced_focal', loss_weight=1.0, fg_weight=5,
                        bg_weight=1, alpha=1, gamma=2)).eval()
    head.depth_samples = O.depth_samples(cfg)
    head.downsample_factor = 4
    with torch.no_grad():
        cost, stereo, mono = m(cur, prev, copy.deepcopy(metas))
        volume = ns.build_dfm_cost(
            cur, prev, m.downsampled_depth, 1, 4,
            torch.as_tensor(np.array([metas[0]['ori_cam2img']]),
                            dtype=torch.float32),
            metas[0]['cur2prevs'], metas[0]['ori_shape'][:2], flip,
            metas[0]['crop_offset'], img_scale_factor=scale)
        _, sm, preds = head(cost)
    np.savez_compressed(
        os.path.join(HERE, name + '.npz'), cur=cur.numpy(), prev=prev.numpy(),
        volume=volume.numpy().astype(np.float32), cost=cost.numpy(),
        stereo=stereo.numpy(), mono=mono.numpy(), depth_preds=preds.numpy(),
        softmax_slice=sm[0, 0, :, ::8, ::8].numpy())
    print(name, 'cost', tuple(cost.shape), float(cost.abs().max()))


def neck_case(ns):
    rng = np.random.RandomState(21)
    c0, cout, t = 64, 256, 2
    nx, ny, nz = 6, 5, 12
    for name, mod in (('neck_dfm', ns.DfMNeck(c0, cout, num_frames=t)),
                      ('neck_imvoxel', ns.OutdoorImVoxelNeck(c0, cout))):
        mod = mod.eval()
        sd = syn.make_neck_params(rng, mod.state_dict())
        mod.load_state_dict(sd, strict=True)
        cin = c0 * t if name == 'neck_dfm' else c0
        x = torch.from_numpy(
            rng.standard_normal((1, cin, nx, ny, nz)).astype(np.float32))
        with torch.no_grad():
            y = mod(x)[0]
        np.savez_compressed(os.path.join(HERE, name + '.npz'), x=x.numpy(),
                            y=y.numpy(), seed=21)
        print(name, tuple(y.shape), float(y.abs().max()))


def neck_multitile_case(ns):
    """Same two necks on a grid of 3 x 3 tiles (16 x 8 voxels each in the CUDA kernel) with
    ragged edges, so tile seams, the K-outer group loop across tiles and the stride-(1,1,2)
    layers on a multi-tile grid are pinned to the reference.  Inputs regenerate from the
    seed (tests/util.py:make_neck_mt_case); the fixture stores the reference output and a
    checksum of the input."""
    from tests.util import make_neck_mt_case
    for name, make in (('neck_dfm_mt', lambda: ns.DfMNeck(64, 256, num_frames=2)),
                       ('neck_imvoxel_mt', lambda: ns.OutdoorImVoxelNeck(64, 256))):
        rng, x = make_neck_mt_case(name)
        mod = make().eval()
        sd = syn.make_neck_params(rng, mod.state_dict())
        mod.load_state_dict(sd, strict=True)
        with torch.no_grad():
            y = mod(x)[0]
        np.savez_compressed(os.path.join(HERE, name + '.npz'), y=y.numpy(),
                            x_sum=np.float64(x.double().sum().item()),
                            x_abs=np.float64(x.double().abs().sum().item()))
        print(name, tuple(x.shape), '->', tuple(y.shape), float(y.abs().max()))


def bev_stage_case(ns):
    """SURVEY.md section 8(f) row 3 / north_star's "3D box regressions": the reference
    BEVHourglass (verbatim) + LIGAAnchor3DHead._init_layers / forward_single (verbatim method
    bodies) on a synthetic voxel feature; inputs regenerate from the seed."""
    c = syn.make_bev_case(**syn.BEV_CASE)
    gn = dict(type='GN', num_groups=32, requires_grad=True)
    bev = ns.BEVHourglass(160, 64, norm_cfg=gn).eval()
    head = ns.LIGAAnchor3DHead(3, 64, 64, 6, norm_cfg=gn).eval()
    bev.load_state_dict(c['bev'], strict=True)
    head.load_state_dict(c['head'], strict=True)
    v = c['volume']
    with torch.no_grad():
        x = v.view(-1, v.shape[1] * v.shape[2], v.shape[3], v.shape[4])   # dfm.py:427-428
        prehg, feat = bev(x)
        cls, box, dirc = head.forward_single(feat)
    np.savez_compressed(os.path.join(HERE, 'bev_stage.npz'), prehg=prehg.numpy(),
                        bev=feat.numpy(), cls_score=cls.numpy(), bbox_pred=box.numpy(),
                        dir_cls_preds=dirc.numpy(),
                        x_sum=np.float64(v.double().sum().item()))
    print('bev_stage', tuple(cls.shape), tuple(box.shape), tuple(dirc.shape),
          float(box.abs().max()))


FRUSTUM_CASE = dict(seed=31, h=32, w=64, num_planes=8, n_voxels=(24, 20, 8))


def frustum_case(ns):
    """Reference DepthHead + FrustumToVoxel run verbatim on the synthetic case
    (the reference calls .cuda() on its voxel grid: made a no-op on this CPU box)."""
    c = syn.make_frustum_case(**FRUSTUM_CASE)
    cfg = c['depth_cfg']
    head = ns.DepthHead(
        depth_cfg=dict(mode='UD', num_bins=cfg['num_bins'], min_depth=2,
                       max_depth=59.6), with_convs=False, num_views=1,
        depth_loss=dict(type='balanced_focal', loss_weight=1.0, fg_weight=5,
                        bg_weight=1, alpha=1, gamma=2)).eval()
    head.depth_samples = O.depth_samples(cfg)
    head.downsample_factor = 4
    m = ns.FrustumToVoxel().eval()
    m.load_state_dict(c['params'], strict=True)
    m.coordinates_3d = c['coordinates_3d']
    m.depth_cfg = cfg
    saved = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        with torch.no_grad():
            _, sm, _ = head(c['cost'])
            out = m(c['stereo'], sm, copy.deepcopy(c['metas']), c['sem'])
    finally:
        torch.Tensor.cuda = saved
    np.savez_compressed(
        os.path.join(HERE, 'frustum.npz'), stereo=c['stereo'].numpy(),
        cost=c['cost'].numpy(), sem=c['sem'].numpy(), softmax=sm.numpy(),
        out=out.numpy())
    print('frustum', tuple(out.shape), float(out.abs().max()),
          float((out != 0).float().mean()))


def state_dict_layout_case(ns):
    """Key order and shapes of the reference modules' state_dicts (the on-disk checkpoint
    contract the mirrors in depth_from_motion_b200/modules.py must keep)."""
    from tests.util import STATE_DICT_MODULES
    layout = {name: [[k, list(v.shape)] for k, v in make(ns).state_dict().items()]
              for name, make in STATE_DICT_MODULES.items()}
    with open(os.path.join(HERE, 'state_dict_layout.json'), 'w') as f:
        json.dump(layout, f, indent=0)
        f.write('\n')
    print('state_dict_layout', {k: len(v) for k, v in layout.items()})


def config_blocks_case(ref_root):
    """The hot-path blocks of the `model` dict of each shipped configs/dfm/*.py, as parsed."""
    from depth_from_motion_b200 import registry
    from tests.util import CONFIG_MODEL_BLOCKS, DFM_CONFIGS
    out = {}
    for name in DFM_CONFIGS:
        model = registry.Config.fromfile(os.path.join(ref_root, 'configs/dfm', name)).model
        out[name] = {k: model[k] for k in CONFIG_MODEL_BLOCKS[model['type']]}
    with open(os.path.join(HERE, 'config_model_blocks.json'), 'w') as f:
        json.dump(out, f, indent=1)
        f.write('\n')
    print('config_model_blocks', {k: sorted(v) for k, v in out.items()})


def voxel_sample_case(ns):
    """The reference voxel_sample (point_fusion.py:324-410, executed verbatim) on the inputs
    of tests/util.py:voxel_sample_args."""
    import torch.nn.functional as F
    from oracle.ref_loader import reference_function
    from tests.util import voxel_sample_args
    ref = reference_function('mmdet3d/models/fusion_layers/point_fusion.py', 'voxel_sample',
                             dict(torch=torch, F=F, points_img2cam=ns.points_img2cam))
    out = {}
    for flip, aligned in ((False, True), (True, True), (False, False)):
        out[f'flip{int(flip)}_aligned{int(aligned)}'] = \
            ref(*voxel_sample_args(flip), aligned=aligned).numpy()
    np.savez_compressed(os.path.join(HERE, 'voxel_sample.npz'), **out)
    print('voxel_sample', {k: v.shape for k, v in out.items()})


def bev_stage_small_case(ns):
    """Reference BEVHourglass + LIGAAnchor3DHead.forward_single on tests/util.py:BEV_SMALL_CASE
    (a 12 x 16 BEV grid)."""
    from tests.util import BEV_SMALL_CASE
    c = syn.make_bev_case(**BEV_SMALL_CASE)
    gn = dict(type='GN', num_groups=32, requires_grad=True)
    bev = ns.BEVHourglass(160, 64, norm_cfg=gn).eval()
    head = ns.LIGAAnchor3DHead(3, 64, 64, 6, norm_cfg=gn).eval()
    bev.load_state_dict(c['bev'], strict=True)
    head.load_state_dict(c['head'], strict=True)
    with torch.no_grad():
        _, feat = bev(c['volume'].reshape(1, 160, 12, 16))
        cls, box, dirc = head.forward_single(feat)
    np.savez_compressed(os.path.join(HERE, 'bev_stage_small.npz'), cls_score=cls.numpy(),
                        bbox_pred=box.numpy(), dir_cls_preds=dirc.numpy())
    print('bev_stage_small', tuple(cls.shape), tuple(box.shape), tuple(dirc.shape))


def spp_lastconv_case(ns):
    """Reference SPPUNetNeck.lastconv (spp_unet_neck.py:60-75, :110): its parameters as the
    reference initialises them, and its output on tests/util.py:spp_lastconv_input."""
    from tests.util import spp_lastconv_input
    gn = dict(type='GN', num_groups=32, requires_grad=True)
    m = ns.SPPUNetNeck(in_channels=[3, 64, 128, 128, 128], start_level=2, sem_channels=[128, 32],
                       stereo_channels=[32, 32], with_upconv=True, cat_img_feature=True,
                       norm_cfg=gn).eval()
    p = {k: v.numpy() for k, v in m.state_dict().items() if k.startswith('lastconv')}
    with torch.no_grad():
        y = m.lastconv(spp_lastconv_input())
    np.savez_compressed(os.path.join(HERE, 'spp_unet_lastconv.npz'), y=y.numpy(), **p)
    print('spp_unet_lastconv', sorted(p), tuple(y.shape))


def pipeline_meta_case(ref_root):
    """The reference VideoPipeline (loading.py) on the geometry of its demo KITTI sample, and
    RandomCrop3D._crop_data (transforms_3d.py), both executed verbatim."""
    import pickle
    from oracle.ref_loader import reference_class
    with open(os.path.join(ref_root, 'demo/data/kitti/kitti_000008_infos.pkl'), 'rb') as f:
        info = pickle.load(f)[0]
    img_info = dict(filename='x.png', cam2global=info['image']['cam2global'],
                    sweeps=[dict(data_path=s['data_path'], cam2global=s['cam2global'])
                            for s in info['image']['sweeps']])

    class Compose:   # the image transforms are out of scope: identity
        def __init__(self, t):
            pass

        def __call__(self, r):
            r['img'] = 0
            return r

    VP = reference_class('mmdet3d/datasets/pipelines/loading.py', 'VideoPipeline',
                         dict(np=np, copy=copy, Compose=Compose))
    out = dict(cam2global=np.asarray(img_info['cam2global'], np.float64),
               sweep_cam2global=np.stack([s['cam2global'] for s in img_info['sweeps']]),
               sweep_paths=np.array([s['data_path'] for s in img_info['sweeps']]))
    for nref, rand in ((1, False), (3, False), (2, True)):
        np.random.seed(7)
        ref = VP([], num_ref_imgs=nref, random=rand)(dict(img_info=copy.deepcopy(img_info)))
        out[f'cur2prevs_n{nref}_random{int(rand)}'] = np.asarray(ref['cur2prevs'])

    class RandomCrop:   # mmdet base: only what _crop_data touches
        def __init__(self, **kw):
            self.bbox_clip_border = kw.get('bbox_clip_border', True)
            self.bbox2label, self.bbox2mask = {}, {}

    RC = reference_class('mmdet3d/datasets/pipelines/transforms_3d.py', 'RandomCrop3D',
                         dict(np=np, RandomCrop=RandomCrop))
    rc = RC(crop_size=(320, 1280), rel_offset_h=(0.3, 1.0))
    img = np.zeros((375, 1242, 3), dtype=np.uint8)
    np.random.seed(3)
    ref = rc._crop_data(dict(img=img, cam2img=syn.KITTI_P2.copy()), (320, 1280), True)
    out.update(crop_offset=np.asarray(ref['crop_offset']),
               crop_cam2img=np.asarray(ref['cam2img'], np.float64),
               crop_img_shape=np.asarray(ref['img_shape']))
    np.savez_compressed(os.path.join(HERE, 'pipeline_meta.npz'), **out)
    print('pipeline_meta', {k: v.shape for k, v in out.items()})


def reference_checks(ns):
    from oracle.ref_loader import REFERENCE_ROOT
    state_dict_layout_case(ns)
    config_blocks_case(REFERENCE_ROOT)
    voxel_sample_case(ns)
    bev_stage_small_case(ns)
    spp_lastconv_case(ns)
    pipeline_meta_case(REFERENCE_ROOT)


def main():
    from tests.util import FIXTURE_THREADS
    ns = load_reference()
    torch.manual_seed(0)
    torch.set_num_threads(FIXTURE_THREADS)
    if 'frustum' in sys.argv[1:]:
        frustum_case(ns)
        return
    if 'bev' in sys.argv[1:]:
        bev_stage_case(ns)
        return
    if 'neck_mt' in sys.argv[1:]:
        neck_multitile_case(ns)
        return
    if 'checks' in sys.argv[1:]:
        reference_checks(ns)
        return
    for name, spec in KITTI_CASES.items():
        kitti_case(ns, name, spec)
    neck_case(ns)
    neck_multitile_case(ns)
    frustum_case(ns)
    bev_stage_case(ns)
    reference_checks(ns)


if __name__ == '__main__':
    main()
