"""CPU tests of the input-side metadata (SURVEY.md section 8(f) row 4) against the reference's
own VideoPipeline / RandomCrop3D code executed verbatim on the demo KITTI sample."""
import os

import numpy as np

from depth_from_motion_b200 import pipeline_meta as pm
from depth_from_motion_b200 import synthetic as syn
from tests.util import GOLDEN


def test_cur2prevs_matches_recorded_demo_geometry():
    # the constants in synthetic.py were read from the demo sample through this very formula
    c2p = syn.KITTI_CUR2PREV
    cur = np.eye(4)
    prevs = [np.linalg.inv(m) for m in c2p]      # prev_cam2global with cur at the origin
    out = pm.cur2prevs(cur, prevs)
    assert out.shape == (3, 4, 4)
    assert np.allclose(out, c2p, atol=1e-9)


def test_select_ref_frames_modes():
    assert pm.select_ref_frames(3, 1, random=False).tolist() == [2]      # test: the last one
    assert pm.select_ref_frames(3, 2, random=False).tolist() == [1, 2]
    assert pm.select_ref_frames(3, -1).size == 0 and pm.select_ref_frames(0, 2).size == 0
    rng = np.random.RandomState(0)
    ids = pm.select_ref_frames(3, 5, random=True, rng=rng)               # with replacement
    assert len(ids) == 5 and set(ids.tolist()) <= {0, 1, 2}


def test_quaternion_matrix():
    m = pm.quaternion_matrix([np.cos(0.3), 0, 0, np.sin(0.3)])          # yaw 0.6 rad
    assert np.allclose(m[:2, :2], [[np.cos(0.6), -np.sin(0.6)], [np.sin(0.6), np.cos(0.6)]])
    assert np.allclose(m[:3, :3] @ m[:3, :3].T, np.eye(3))


def test_video_meta_matches_reference_pipeline():
    """Against the reference VideoPipeline executed verbatim on the geometry of its demo KITTI
    sample (both stored in tests/golden/pipeline_meta.npz)."""
    gold = np.load(os.path.join(GOLDEN, 'pipeline_meta.npz'))
    img_info = dict(filename='x.png', cam2global=gold['cam2global'],
                    sweeps=[dict(data_path=str(p), cam2global=m)
                            for p, m in zip(gold['sweep_paths'], gold['sweep_cam2global'])])
    for nref, rand in ((1, False), (3, False), (2, True)):
        ref = gold[f'cur2prevs_n{nref}_random{int(rand)}']
        got = pm.video_meta(img_info, nref, rand, rng=np.random.RandomState(7))
        assert np.array_equal(ref, got['cur2prevs'])
        assert [m for m in got['ref_filenames']] == \
            [img_info['sweeps'][i]['data_path'] for i in got['ref_ids']]
    # the three sweeps are what synthetic.KITTI_CUR2PREV records (nearest first)
    allp = pm.video_meta(img_info, 3, False)['cur2prevs']
    assert np.allclose(allp, syn.KITTI_CUR2PREV, atol=1e-6)


def test_crop3d_meta_matches_reference():
    """Against RandomCrop3D._crop_data executed verbatim (crop (320, 1280) of a 375 x 1242
    image, np.random.seed(3); stored in tests/golden/pipeline_meta.npz)."""
    gold = np.load(os.path.join(GOLDEN, 'pipeline_meta.npz'))
    rng = np.random.RandomState(3)
    x1, y1 = pm.random_crop_offsets((375, 1242, 3), (320, 1280), (0.3, 1.0), (0., 1.), rng)
    cam, off = pm.crop3d_meta(syn.KITTI_P2, x1, y1)
    assert off == gold['crop_offset'].tolist()
    assert np.allclose(cam, gold['crop_cam2img'], atol=1e-9)
    assert tuple(gold['crop_img_shape'][:2].tolist()) == (320, 1242)


def test_backbone_img_meta_feeds_geometry_packing():
    from depth_from_motion_b200 import modules
    c2p = pm.cur2prevs(np.eye(4), [np.linalg.inv(syn.KITTI_CUR2PREV[2])])
    meta = pm.backbone_img_meta(syn.KITTI_P2, c2p, (375, 1242, 3), (320, 1280, 3),
                                crop_offset=(0, 55))
    g = modules.geometry_from_meta(meta)
    assert abs(g.cur2prev[11] - syn.KITTI_CUR2PREV[2][2, 3]) < 1e-6
    assert (g.crop_x, g.crop_y) == (0.0, 55.0) and g.org_w == 1242
