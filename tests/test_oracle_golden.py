"""CPU tests: the oracle restatement against (1) the reference's own golden vectors
for this path (SURVEY.md section 8c) and (2) fixtures produced by the unmodified
reference sources (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from depth_from_motion_b200 import synthetic as syn
from oracle import dfm_oracle as O
from tests.util import FIXTURE_THREADS, GOLDEN, KITTI_CASES, load_kitti_case


@pytest.fixture(autouse=True)
def _fixture_threads():
    """The CPU kernels split their reductions (float64 sums, convolutions) by the number of
    intra-op threads, so the oracle reproduces the fixtures to the bit only with the thread
    count they were generated with, whatever the host's core count."""
    saved = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(saved)


def test_points_img2cam_kat():
    # reference tests/test_utils/test_utils.py:186-193
    points = torch.tensor([[0.5764, 0.9109, 0.7576], [0.6656, 0.5498, 0.9813]])
    cam2img = torch.tensor([[700., 0., 450., 0.], [0., 700., 200., 0.],
                            [0., 0., 1., 0.]])
    expected = torch.tensor([[-0.4864, -0.2155, 0.7576],
                             [-0.6299, -0.2796, 0.9813]])
    assert torch.allclose(O.points_img2cam(points, cam2img), expected, atol=1e-3)


def test_points_cam2img_kat():
    # reference tests/test_utils/test_box3d.py:1653-1680
    torch.manual_seed(0)
    points = torch.rand([5, 3])
    proj_mat = torch.rand([4, 4])
    expected = torch.tensor([[0.5832, 0.6496], [0.6146, 0.7910],
                             [0.6994, 0.7782], [0.5623, 0.6303],
                             [0.4359, 0.6532]])
    assert torch.allclose(O.points_cam2img(points, proj_mat), expected, 1e-3)
    expected_d = torch.tensor([[0.5832, 0.6496, 1.7577], [0.6146, 0.7910, 1.5477],
                               [0.6994, 0.7782, 2.0091], [0.5623, 0.6303, 1.8739],
                               [0.4359, 0.6532, 1.2056]])
    assert torch.allclose(O.points_cam2img(points, proj_mat, with_depth=True),
                          expected_d, 1e-3)


def test_point_sample_kat():
    # reference tests/test_models/test_fusion/test_point_fusion.py:13-41 (the
    # no-3D-augmentation half; PointFusion.sample_single -> point_sample with
    # scale 1, crop 0, no flip, bilinear, align_corners=True)
    lidar2img = torch.tensor(
        [[6.0294e+02, -7.0791e+02, -1.2275e+01, -1.7094e+02],
         [1.7678e+02, 8.8088e+00, -7.0794e+02, -1.0257e+02],
         [9.9998e-01, -1.5283e-03, -5.2907e-03, -3.2757e-01],
         [0.0000e+00, 0.0000e+00, 0.0000e+00, 1.0000e+00]])
    img_feat = torch.arange(370 * 1224)[None, ...].view(
        370, 1224)[None, None, ...].float() / (370 * 1224)
    pts = torch.tensor([[8.356, -4.312, -0.445], [11.777, -6.724, -0.564],
                        [6.453, 2.53, -1.612], [6.227, -3.839, -0.563]])
    out = O.point_sample(img_feat, pts, lidar2img, pts.new_tensor([1., 1.]),
                         0, False, (370, 1224), (370, 1224), aligned=True)
    expected = torch.tensor([0.5560822, 0.5476625, 0.9687978, 0.6241757])
    assert torch.allclose(expected, out.squeeze(), 1e-4)


@pytest.mark.parametrize('name', sorted(KITTI_CASES))
def test_backbone_matches_reference_fixture(name):
    cur, prev, metas, params, cfg, gold = load_kitti_case(name)
    spec = KITTI_CASES[name]
    with torch.no_grad():
        vol = O.build_dfm_cost(
            cur, prev, O.downsampled_depth(cfg), 1, 4,
            torch.as_tensor(np.array([metas[0]['ori_cam2img']]),
                            dtype=torch.float32), metas[0]['cur2prevs'],
            metas[0]['ori_shape'][:2], spec[4], metas[0]['crop_offset'],
            img_scale_factor=spec[6])
        cost, stereo, mono = O.dfm_backbone_forward(params, cur, prev, metas, cfg)
        _, sm, preds = O.depth_head_forward(cost, O.depth_samples(cfg))
    # same ATen ops, same order, same machine class: tiny tolerance only for
    # thread-count dependent summation order
    for got, key in ((vol, 'volume'), (cost, 'cost'), (stereo, 'stereo'),
                     (mono, 'mono'), (preds, 'depth_preds')):
        ref = torch.from_numpy(gold[key])
        assert got.shape == ref.shape, key
        assert torch.allclose(got, ref, rtol=1e-4, atol=1e-5), key
    assert torch.allclose(sm[0, 0, :, ::8, ::8],
                          torch.from_numpy(gold['softmax_slice']), atol=1e-6)


def test_generated_inputs_match_stored_inputs():
    # fixture inputs regenerate bit-identically from their seed
    for name, spec in KITTI_CASES.items():
        seed, h, w, d = spec[:4]
        cur, prev, _, _ = syn.make_kitti_pair(seed, h, w, d)
        gold = np.load(os.path.join(GOLDEN, name + '.npz'))
        assert np.array_equal(cur.numpy(), gold['cur'])
        assert np.array_equal(prev.numpy(), gold['prev'])


@pytest.mark.parametrize('name', ['neck_dfm', 'neck_imvoxel'])
def test_neck_matches_reference_fixture(name):
    from depth_from_motion_b200 import modules
    gold = np.load(os.path.join(GOLDEN, name + '.npz'))
    rng = np.random.RandomState(21)
    dfm = modules.DfMNeck(64, 256, num_frames=2)
    imv = modules.OutdoorImVoxelNeck(64, 256)
    # make_golden draws the DfMNeck parameters first, then its input, then the
    # OutdoorImVoxelNeck parameters: replay the same stream
    sd_dfm = syn.make_neck_params(rng, dfm.state_dict())
    x_dfm = rng.standard_normal((1, 128, 6, 5, 12)).astype(np.float32)
    sd_imv = syn.make_neck_params(rng, imv.state_dict())
    x = torch.from_numpy(gold['x'])
    if name == 'neck_dfm':
        assert np.array_equal(x_dfm, gold['x'])
        with torch.no_grad():
            y = O.dfm_neck_forward(sd_dfm, x, 64)[0]
    else:
        with torch.no_grad():
            y = O.imvoxel_neck_forward(sd_imv, x)[0]
    assert torch.allclose(y, torch.from_numpy(gold['y']), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('name', ['neck_dfm_mt', 'neck_imvoxel_mt'])
def test_neck_multitile_fixture(name):
    """The multi-tile neck fixtures (37 x 21 x 12 voxels = 3 x 3 tiles of the CUDA kernel,
    ragged edges): inputs regenerate from the seed (checksums stored), the oracle restatement
    reproduces the verbatim reference output."""
    from depth_from_motion_b200 import modules
    from tests.util import make_neck_mt_case
    gold = np.load(os.path.join(GOLDEN, name + '.npz'))
    rng, x = make_neck_mt_case(name)
    assert float(x.double().sum()) == float(gold['x_sum'])
    assert float(x.double().abs().sum()) == float(gold['x_abs'])
    mod = (modules.DfMNeck(64, 256, num_frames=2) if name == 'neck_dfm_mt'
           else modules.OutdoorImVoxelNeck(64, 256))
    sd = syn.make_neck_params(rng, mod.state_dict())
    with torch.no_grad():
        y = (O.dfm_neck_forward(sd, x, 64) if name == 'neck_dfm_mt'
             else O.imvoxel_neck_forward(sd, x))[0]
    ref = torch.from_numpy(gold['y'])
    assert y.shape == ref.shape == (1, 256, 21, 37)
    assert torch.allclose(y, ref, rtol=1e-4, atol=1e-4)


def test_depth_tables():
    cfg = syn.depth_cfg_for(72)
    d = O.downsampled_depth(cfg)
    assert d.shape == (72,) and abs(float(d[0]) - (2 + 0.5 * 4 * 0.2)) < 1e-5
    s = O.depth_samples(cfg)
    assert s.shape == (288,) and abs(float(s[-1]) - (59.6 - 0.1)) < 1e-4


def test_frustum_to_voxel_matches_reference_fixture():
    """SURVEY.md section 8(f) row 1: oracle restatement (DepthHead -> FrustumToVoxel)
    against the verbatim reference run stored in tests/golden/frustum.npz."""
    from tests.util import load_frustum_case
    c, gold = load_frustum_case()
    cfg = c['depth_cfg']
    _, sm, _ = O.depth_head_forward(c['cost'], O.depth_samples(cfg), 4)
    assert torch.equal(sm, torch.from_numpy(gold['softmax']))
    out = O.frustum_to_voxel_forward(c['params'], c['stereo'], sm, c['metas'], c['sem'],
                                     c['coordinates_3d'], cfg)
    ref = torch.from_numpy(gold['out'])
    assert out.shape == ref.shape == (1, 32, 2, 20, 24)
    assert float((out - ref).abs().max()) <= 1e-6
    # the grid of the shipped config (detectors/dfm.py:174-211)
    full = O.frustum_coordinates_3d(dict(point_cloud_range=syn.KITTI_POINT_CLOUD_RANGE,
                                         voxel_size=syn.KITTI_VOXEL_SIZE))
    assert tuple(full.shape) == (20, 304, 288, 3)
    assert torch.equal(full, syn.frustum_coordinates(syn.KITTI_POINT_CLOUD_RANGE,
                                                     (288, 304, 20)))


@pytest.mark.parametrize('flip,aligned', [(False, True), (True, True), (False, False)])
def test_voxel_sample_matches_reference_source(flip, aligned):
    """SURVEY.md row a8 (oracle only): the restatement against the reference function executed
    verbatim (point_fusion.py:324-410), stored in tests/golden/voxel_sample.npz."""
    from tests.util import voxel_sample_args
    gold = np.load(os.path.join(GOLDEN, 'voxel_sample.npz'))
    a = torch.from_numpy(gold[f'flip{int(flip)}_aligned{int(aligned)}'])
    b = O.voxel_sample(*voxel_sample_args(flip), aligned=aligned)
    assert a.shape == b.shape == (1, 6, 4, 8, 16)
    assert torch.equal(a, b)
    assert float(a.abs().sum()) > 0


def test_bev_stage_matches_reference_fixture():
    """SURVEY.md section 8(f) row 3: oracle restatement of BEVHourglass + LIGAAnchor3DHead
    (class scores, 3-D box regressions, direction logits) against the verbatim reference run."""
    gold = np.load(os.path.join(GOLDEN, 'bev_stage.npz'))
    c = syn.make_bev_case(**syn.BEV_CASE)
    assert float(c['volume'].double().sum()) == float(gold['x_sum'])
    v = c['volume']
    with torch.no_grad():
        prehg, bev = O.bev_hourglass_forward(c['bev'], v.reshape(1, -1, v.shape[3], v.shape[4]))
        outs = O.dfm_bev_stage(c['bev'], c['head'], v)
    for got, key in ((prehg, 'prehg'), (bev, 'bev'), (outs[0], 'cls_score'),
                     (outs[1], 'bbox_pred'), (outs[2], 'dir_cls_preds')):
        ref = torch.from_numpy(gold[key])
        assert got.shape == ref.shape, key
        assert torch.allclose(got, ref, rtol=1e-4, atol=1e-5), key
    assert outs[0].shape[1] == 18 and outs[1].shape[1] == 42 and outs[2].shape[1] == 12


def test_bev_stage_oracle_equals_reference_source():
    """Bit-for-bit against the reference classes executed verbatim on a 12 x 16 BEV grid
    (tests/golden/bev_stage_small.npz)."""
    from tests.util import BEV_SMALL_CASE
    gold = np.load(os.path.join(GOLDEN, 'bev_stage_small.npz'))
    c = syn.make_bev_case(**BEV_SMALL_CASE)
    with torch.no_grad():
        got = O.dfm_bev_stage(c['bev'], c['head'], c['volume'])
    for a, key in zip(got, ('cls_score', 'bbox_pred', 'dir_cls_preds')):
        assert torch.equal(a, torch.from_numpy(gold[key])), key


def test_spp_unet_lastconv_equals_reference_module():
    """SURVEY.md section 8(f) row 2: the oracle restatement of SPPUNetNeck.lastconv against the
    reference class executed verbatim (spp_unet_neck.py:60-75, :110): its parameters and output
    are stored in tests/golden/spp_unet_lastconv.npz."""
    from tests.util import spp_lastconv_input
    gold = dict(np.load(os.path.join(GOLDEN, 'spp_unet_lastconv.npz')))
    y = torch.from_numpy(gold.pop('y'))
    p = {k: torch.from_numpy(v) for k, v in gold.items()}
    assert sorted(p) == ['lastconv.0.conv.weight', 'lastconv.0.gn.bias', 'lastconv.0.gn.weight',
                         'lastconv.1.weight']
    x = spp_lastconv_input()
    with torch.no_grad():
        assert torch.equal(y, O.spp_unet_lastconv(p, x))
    # the mirror takes the same keys
    from depth_from_motion_b200 import modules
    modules.SPPUNetNeckTail().load_state_dict(p, strict=True)
