"""init='mst' host algorithm (SURVEY §8f rank 1): CPU tests of the spanning-tree / Procrustes / PnP initialiser."""
import copy

import numpy as np
import pytest
import torch

from conftest import digest, reference_records
from dust3r_b200.utils.synth import synth_consistent_scene


def _edges(n):
    e = [(i, j) for i in range(n) for j in range(i)]
    return e + [(j, i) for i, j in e]


def test_mst_init_recovers_consistent_scene():
    """On an exactly consistent scene the initialiser alone must nearly zero the objective's residuals: the
    world pointmaps of every image agree with each aligned pairwise prediction."""
    from dust3r_b200.cloud_opt import global_aligner
    from dust3r_b200.cloud_opt import init_im_poses as init_fun
    from dust3r_b200.utils.geometry import geotrf
    n, H, W = 4, 24, 32
    out, cams, f = synth_consistent_scene(n, _edges(n), H, W, seed=1, noise=0.0)
    import cv2
    cv2.setRNGSeed(0)
    torch.manual_seed(0)
    net = global_aligner(copy.deepcopy(out), 'cpu', verbose=False)
    init_fun.minimum_spanning_tree  # noqa
    pts3d, msp_edges, im_focals, im_poses = init_fun.minimum_spanning_tree(
        net.imshapes, net.edges, net.pred_i, net.pred_j, net.conf_i, net.conf_j, net.im_conf, net.min_conf_thr, 'cpu',
        has_im_poses=True, verbose=False)
    assert len(msp_edges) == n - 1
    assert all(abs(fo - f) / f < 0.05 for fo in im_focals)
    # relative geometry: pairwise camera-centre distances match the ground truth up to one global scale
    c_est = im_poses[:, :3, 3]
    c_gt = cams[:, :3, 3]
    d_est = torch.cdist(c_est, c_est)
    d_gt = torch.cdist(c_gt, c_gt)
    s = (d_est.sum() / d_gt.sum())
    assert torch.allclose(d_est, s * d_gt, atol=0.05 * float(d_gt.max()) * float(s))


def test_mst_init_matches_reference():
    """Same inputs, same cv2 RNG seed -> same initial parameters as the reference initialiser
    (reference cloud_opt + local roma restatement; its parameters recorded in tests/golden/reference_records.npz)."""
    import cv2
    from dust3r_b200.cloud_opt import global_aligner
    import dust3r_b200.cloud_opt.init_im_poses as init_fun
    gold = reference_records()
    n, H, W = 4, 24, 32
    out, cams, f = synth_consistent_scene(n, _edges(n), H, W, seed=2, noise=0.005)

    torch.manual_seed(3)
    cv2.setRNGSeed(0)
    net = global_aligner(copy.deepcopy(out), 'cpu', verbose=False)
    pts3d, _, im_focals, im_poses = init_fun.minimum_spanning_tree(
        net.imshapes, net.edges, net.pred_i, net.pred_j, net.conf_i, net.conf_j, net.im_conf, net.min_conf_thr, 'cpu',
        has_im_poses=True, niter_PnP=10, verbose=False)
    # init_from_pts3d ends with a loss evaluation, which needs the GPU kernel; set parameters only
    net.verbose = False
    try:
        init_fun.init_from_pts3d(net, pts3d, im_focals, im_poses)
    except Exception as e:  # pragma: no cover
        raise
    for k in ('pw_poses', 'im_poses', 'im_focals'):
        a, b = torch.from_numpy(gold[f'mst|{k}']), getattr(net, k).data
        if k.endswith('poses'):   # quaternion sign is arbitrary
            qa, qb = a[:, :4], b[:, :4]
            sign = torch.sign((qa * qb).sum(-1, keepdim=True))
            b = torch.cat((qb * sign, b[:, 4:]), dim=-1)
        assert torch.allclose(a, b, atol=2e-3, rtol=2e-3), (k, float((a - b).abs().max()))
    assert torch.allclose(torch.from_numpy(gold['mst|im_depthmaps']), net.im_depthmaps.data, atol=2e-3, rtol=2e-3)


def test_pair_viewer_matches_live_reference():
    """GlobalAlignerMode.PairViewer (closed form, cv2 PnP) against what the unmodified reference class returns on a consistent
    two-view scene, OpenCV's RANSAC seeded identically (recorded in tests/golden/reference_records.npz; the pointmaps at a
    fixed quarter of the pixels)."""
    import cv2
    from dust3r_b200.cloud_opt import global_aligner as ours, GlobalAlignerMode as OurMode
    gold = reference_records()
    ref = lambda key: torch.from_numpy(gold[f'pair_viewer|{key}'])
    out, cams, f = synth_consistent_scene(2, [(0, 1), (1, 0)], 48, 64, seed=3, noise=0.002)
    cv2.setRNGSeed(0)
    a = ours(copy.deepcopy(out), 'cpu', mode=OurMode.PairViewer, verbose=False)
    assert torch.allclose(a.get_focals(), ref('get_focals'), rtol=1e-6)
    assert torch.allclose(a.get_im_poses(), ref('get_im_poses'), atol=1e-5)
    assert torch.equal(a.get_principal_points(), ref('get_principal_points'))
    assert torch.allclose(a.get_intrinsics(), ref('get_intrinsics'), rtol=1e-6)
    depths, pts, masks, px = a.get_depthmaps(), a.get_pts3d(), a.get_masks(), ref('px')
    assert len(depths) == len(pts) == len(masks) == 2
    for i in range(2):
        assert torch.allclose(depths[i], ref(f'get_depthmaps|{i}'), atol=1e-5)
        assert torch.allclose(pts[i].reshape(-1, 3)[px], ref(f'get_pts3d|{i}'), atol=1e-5)
        assert torch.equal(masks[i], ref(f'get_masks|{i}'))
    assert np.isnan(a())   # no objective: forward() is NaN like the reference's


def test_is_symmetrized_quirks_match_live_reference():
    """Exhaustive over instance lists of length <= 5 on a two-letter alphabet, including the IndexError the reference
    raises for an odd batch of mirrored couples (the reference's outcomes recorded in tests/golden/reference_records.npz:
    1 / 0 / -1 for True / False / IndexError)."""
    import itertools
    from dust3r_b200.utils.misc import is_symmetrized as mine
    ref = iter(reference_records()['is_symmetrized|outcomes'].tolist())

    def outcome(fn, a, b):
        try:
            return int(bool(fn(dict(instance=a), dict(instance=b))))
        except IndexError:
            return -1
    for n in range(1, 6):
        for a in itertools.product('ab', repeat=n):
            for b in itertools.product('ab', repeat=n):
                assert outcome(mine, list(a), list(b)) == next(ref), (a, b)
    assert next(ref, None) is None


@pytest.mark.parametrize('fx_and_fy', [False, True])
def test_modular_optimizer_presets_match_live_reference(fx_and_fy):
    """Host-side API of ModularPointCloudOptimizer (presets with int / list / boolean-tensor / array masks, parameter
    encodings, intrinsics, world pointmaps) against what the unmodified reference class returns, same seeds, on the CPU
    (recorded in tests/golden/reference_records.npz; the pointmaps and depthmaps as digests)."""
    import warnings
    warnings.filterwarnings('ignore')
    from dust3r_b200.utils.synth import synth_pair_predictions
    from dust3r_b200.cloud_opt import global_aligner as ours, GlobalAlignerMode as OurMode
    gold = reference_records()
    ref = lambda key: gold[f'modular|{int(fx_and_fy)}|{key}']
    n, H, W = 4, 24, 32
    edges = [(i, j) for i in range(n) for j in range(n) if i != j]
    out = synth_pair_predictions(n, edges, H, W, seed=2)
    torch.manual_seed(0)
    a = ours(copy.deepcopy(out), 'cpu', mode=OurMode.ModularPointCloudOptimizer, verbose=False, fx_and_fy=fx_and_fy, optimize_pp=True)
    Ks = [torch.tensor([[30. + i, 0, 15 + i], [0, 32. + i, 11 - i], [0, 0, 1.]]) for i in range(2)]
    poses = [torch.eye(4), torch.tensor([[0., -1, 0, 1], [1, 0, 0, 2], [0, 0, 1, 3], [0, 0, 0, 1]])]
    a.preset_intrinsics(Ks, msk=[1, 3])
    a.preset_pose(poses, pose_msk=torch.tensor([True, False, True, False]))
    a.preset_focal([55.0], msk=0)
    a.preset_principal_point([torch.tensor([14., 13.])], msk=np.array([2]))
    assert a.norm_pw_scale == bool(ref('norm_pw_scale'))
    for name in ('im_poses', 'im_pp', 'im_focals'):
        assert [p.requires_grad for p in getattr(a, name)] == ref(f'requires_grad|{name}').tolist(), name
    for get in ('get_focals', 'get_principal_points', 'get_intrinsics', 'get_im_poses'):
        assert torch.equal(getattr(a, get)(), torch.from_numpy(ref(get))), get
    assert [digest(x) for x in a.get_pts3d()] == ref('get_pts3d').tolist()
    assert [digest(x) for x in a.get_depthmaps()] == ref('get_depthmaps').tolist()
    assert a.get_known_focal_mask().tolist() == [True, True, False, True]
