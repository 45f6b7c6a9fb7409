"""Shared helpers for the test-suite."""
import os

import numpy as np
import torch

from depth_from_motion_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
# intra-op CPU threads tests/golden/make_golden.py computes the fixtures with
FIXTURE_THREADS = 8

# must match tests/golden/make_golden.py
KITTI_CASES = {
    'kitti_plain': (11, 32, 64, 8, False, (0, 0), 1.0, None),
    'kitti_aug': (12, 32, 64, 8, True, (10, 40), 1.03, (375, 1242, 3)),
}


def load_kitti_case(name):
    seed, h, w, d, flip, crop, scale, ori = KITTI_CASES[name]
    cur, prev, metas, params = syn.make_kitti_pair(
        seed, h, w, d, flip=flip, crop_offset=crop, scale=scale, ori_shape=ori)
    gold = dict(np.load(os.path.join(GOLDEN, name + '.npz')))
    # the stored inputs are authoritative (regeneration is only a convenience)
    cur = torch.from_numpy(gold['cur'])
    prev = torch.from_numpy(gold['prev'])
    return cur, prev, metas, params, syn.depth_cfg_for(d), gold


def rel_err(a, b):
    """max |a-b| / max |b|  -- the normalised max-norm error used for the 1e-3 bar."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def assert_close(a, b, what='', rtol=1e-3, atol_frac=1e-4):
    """Element-wise form of the north_star tolerance ("1e-3 relative fp32"):
    |a - b| <= rtol * |b| + atol_frac * max|b| for EVERY element.  The absolute term only
    covers values that are themselves ~1e-4 of the tensor's scale (zero crossings of a
    feature map have no meaningful relative error); everything else must be within 1e-3 of
    its own magnitude.  Returns the worst ratio |a-b| / (rtol |b| + atol)."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    atol = atol_frac * float(b.abs().max())
    ratio = float(((a - b).abs() / (rtol * b.abs() + atol)).max())
    assert ratio <= 1.0, f'{what}: worst element is {ratio:.2f}x the tolerance'
    return ratio


# must match tests/golden/make_golden.py
NECK_MT_SHAPE = (37, 21, 12)   # (Nx, Ny, Nz): 3 x 3 tiles of the 16 x 8 neck tile, ragged edges
NECK_MT_SEED = 77


def make_neck_mt_case(name):
    """Multi-tile neck fixture inputs, regenerated from the seed (only the reference output and
    input checksums are stored).  Returns (module kwargs, state_dict template filler, x)."""
    rng = np.random.RandomState(NECK_MT_SEED + (0 if name == 'neck_dfm_mt' else 1))
    cin = 128 if name == 'neck_dfm_mt' else 64
    x = torch.from_numpy(rng.standard_normal((1, cin) + NECK_MT_SHAPE).astype(np.float32))
    return rng, x


# must match tests/golden/make_golden.py
FRUSTUM_CASE = dict(seed=31, h=32, w=64, num_planes=8, n_voxels=(24, 20, 8))


def load_frustum_case():
    c = syn.make_frustum_case(**FRUSTUM_CASE)
    gold = dict(np.load(os.path.join(GOLDEN, 'frustum.npz')))
    for k in ('stereo', 'cost', 'sem'):
        c[k] = torch.from_numpy(gold[k])
    return c, gold


# must match tests/golden/make_golden.py: the modules whose state_dict layout (key order and
# shapes) is stored in state_dict_layout.json; `ns` is either the package's `modules` or the
# reference namespace, both have these class names
STATE_DICT_MODULES = {
    'DfMBackbone': lambda ns: ns.DfMBackbone(in_channels=32, depth_cfg=syn.depth_cfg_for(16)),
    'DfMNeck': lambda ns: ns.DfMNeck(64, 256, num_frames=2),
    'OutdoorImVoxelNeck': lambda ns: ns.OutdoorImVoxelNeck(64, 256),
    'FrustumToVoxel': lambda ns: ns.FrustumToVoxel(),
    'FrustumToVoxel(num_3dconvs=2, cat_img_feature=False)':
        lambda ns: ns.FrustumToVoxel(num_3dconvs=2, cat_img_feature=False),
}

# the shipped configs/dfm/*.py and, per detector type, the blocks of their `model` dict that
# the hot path is built from (stored in config_model_blocks.json)
DFM_CONFIGS = ('dfm_r34_1x8_kitti-3d-3class.py',
               'multiview-dfm_r101_dcn_2x16_waymoD5-3d-3class_camsync.py',
               'multiview-dfm_r101_dcn_2x16_waymoD5-3d-3class_camsync_10sweeps.py')
CONFIG_MODEL_BLOCKS = {
    'DfM': ('type', 'depth_cfg', 'voxel_cfg', 'backbone_stereo', 'depth_head',
            'feature_transformation', 'backbone_3d', 'bbox_head_3d'),
    'MultiViewDfM': ('type', 'neck_3d'),
}


def voxel_sample_args(flip):
    """Inputs of the voxel_sample fixture (voxel_sample.npz): a camera looking along +x."""
    g = torch.Generator().manual_seed(3)
    vox = torch.randn(1, 6, 20, 16, 8, generator=g)
    vrange, vsize = [0.0, -8.0, -2.0, 20.0, 8.0, 2.0], [1.0, 1.0, 0.5]
    depths = torch.linspace(2.0, 18.0, 16)
    # lidar -> image: camera looks along +x
    k = torch.tensor([[40., 0, 32, 0], [0, 40., 16, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
    l2c = torch.tensor([[0., -1, 0, 0], [0, 0, -1, 0.3], [1, 0, 0, 0.1], [0, 0, 0, 1]])
    proj = k @ l2c
    return (vox, vrange, vsize, depths, proj, 4, torch.tensor([1.02, 0.98]),
            torch.tensor([1.0, 2.0]), flip, (32, 64), (30, 62))


# must match tests/golden/make_golden.py
BEV_SMALL_CASE = dict(seed=5, nz=5, ny=12, nx=16)


def spp_lastconv_input():
    return torch.randn(1, 32, 24, 40, generator=torch.Generator().manual_seed(4))
