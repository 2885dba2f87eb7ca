"""CPU tests of the host-side mirror of the reference API (no GPU, no compute through the .so)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, digest, reference_records
from dust3r_b200.config import vitl_512_dpt, vitl_224_linear, state_dict_spec
from dust3r_b200.image_pairs import make_pairs


@pytest.mark.parametrize('name,cfg', [('dpt512', vitl_512_dpt()), ('lin224', vitl_224_linear())])
def test_state_dict_layout_matches_reference(name, cfg):
    ref = json.load(open(os.path.join(GOLDEN, f'ref_state_dict_{name}.json')))
    spec = state_dict_spec(cfg)
    assert list(ref.keys()) == list(spec.keys())
    for k in ref:
        assert tuple(ref[k]) == tuple(spec[k]), k


def test_make_pairs_bit_exact_against_reference_golden():
    gold = np.load(os.path.join(GOLDEN, 'make_pairs.npz'))
    assert len(gold.files) == 168
    for key in gold.files:
        n, sg, sym, pf = key.split('|')
        imgs = [dict(idx=i, instance=str(i)) for i in range(int(n))]
        pairs = make_pairs(imgs, scene_graph=sg, prefilter=None if pf == 'None' else pf, symmetrize=bool(int(sym)))
        got = np.int32([(a['idx'], b['idx']) for a, b in pairs]).reshape(-1, 2)
        assert got.shape == gold[key].shape, key
        assert (got == gold[key]).all(), key


def test_make_pairs_counts():
    imgs = [dict(idx=i, instance=str(i)) for i in range(8)]
    assert len(make_pairs(imgs, symmetrize=False)) == 28
    assert len(make_pairs(imgs, symmetrize=True)) == 56
    imgs = [dict(idx=i, instance=str(i)) for i in range(50)]
    assert len(make_pairs(imgs, symmetrize=False)) == 1225


def test_rotation_helpers_roundtrip():
    from dust3r_b200.cloud_opt.commons import unitquat_to_rotmat, rotmat_to_unitquat, rigid_points_registration
    g = torch.Generator().manual_seed(0)
    q = torch.randn((64, 4), generator=g)
    R = unitquat_to_rotmat(q)
    assert torch.allclose(R @ R.transpose(-1, -2), torch.eye(3).expand(64, 3, 3), atol=1e-5)
    q2 = rotmat_to_unitquat(R)
    assert torch.allclose(unitquat_to_rotmat(q2), R, atol=1e-5)
    x = torch.randn((500, 3), generator=g)
    s, t = 1.7, torch.tensor([0.3, -2.0, 1.0])
    y = s * x @ R[0].T + t
    Rr, tr, sr = rigid_points_registration(x, y, weights=torch.rand(500, generator=g) + 0.1, compute_scaling=True)
    assert torch.allclose(Rr, R[0], atol=1e-4) and torch.allclose(tr, t, atol=1e-4) and abs(float(sr) - s) < 1e-4


def test_optimizer_host_objects_on_cpu():
    """Construction, parametrisation and getters work without a GPU; the optimisation itself must
    refuse to run anywhere but on a B200 (no CPU fallback)."""
    from dust3r_b200.cloud_opt import global_aligner, GlobalAlignerMode
    from dust3r_b200.utils.synth import synth_pair_predictions
    from dust3r_b200._lib import D3RError
    n, H, W = 3, 16, 32
    edges = [(i, j) for i in range(n) for j in range(i)]
    out = synth_pair_predictions(n, edges, H, W, seed=2)
    torch.manual_seed(0)
    net = global_aligner(out, 'cpu', mode=GlobalAlignerMode.PointCloudOptimizer, verbose=False)
    assert net.im_depthmaps.shape == (n, H * W) and net.im_poses.shape == (n, 7)
    assert net.im_focals.shape == (n, 1) and net.pw_poses.shape == (len(edges), 8)
    assert abs(float(net.get_focals()[0]) - max(H, W)) < 1e-3
    assert net.get_im_poses().shape == (n, 4, 4)
    assert [tuple(p.shape) for p in net.get_pts3d()] == [(H, W, 3)] * n
    sd = net.state_dict()
    assert set(sd) == {'pw_poses', 'pw_adaptors', 'im_depthmaps', 'im_poses', 'im_focals', 'im_pp'} | {f'im_conf.{i}' for i in range(n)}
    with pytest.raises(D3RError):
        net.compute_global_alignment(init=None, niter=2)
    net2 = global_aligner(out, 'cpu', mode=GlobalAlignerMode.ModularPointCloudOptimizer, verbose=False)
    assert len(net2.im_depthmaps) == n and net2.get_intrinsics().shape == (n, 3, 3)
    # the opt-in early upload is a no-op off CUDA and never reaches the optimizer's constructor; the caller's dict is untouched
    torch.manual_seed(0)
    net3 = global_aligner(out, 'cpu', verbose=False, early_upload=True)
    assert torch.equal(net3.im_depthmaps, net.im_depthmaps) and torch.equal(net3.pw_poses, net.pw_poses)
    assert out['pred1']['pts3d'].device.type == 'cpu'


def test_optimizer_init_matches_reference_draws():
    """Same torch seed -> same initial parameters as the reference constructor (optimizer.py:29-33), whose draws are recorded
    in tests/golden/reference_records.npz."""
    import copy
    from dust3r_b200.cloud_opt import global_aligner, GlobalAlignerMode
    from dust3r_b200.utils.synth import synth_pair_predictions
    gold = reference_records()
    n, H, W = 3, 16, 32
    edges = [(i, j) for i in range(n) for j in range(i)]
    out = synth_pair_predictions(n, edges, H, W, seed=2)
    torch.manual_seed(123)
    net = global_aligner(copy.deepcopy(out), 'cpu', mode=GlobalAlignerMode.PointCloudOptimizer, verbose=False)
    for k in ('pw_poses', 'im_depthmaps', 'im_poses', 'im_focals', 'im_pp'):
        assert torch.equal(torch.from_numpy(gold[f'init_draws|{k}']), getattr(net, k).data), k
    pts = net.get_pts3d()
    assert len(pts) == len([k for k in gold.files if k.startswith('init_draws|pts3d|')])
    for i, b in enumerate(pts):
        assert torch.allclose(torch.from_numpy(gold[f'init_draws|pts3d|{i}']), b, atol=1e-5, rtol=1e-5)
    assert torch.allclose(torch.from_numpy(gold['init_draws|get_pw_poses']), net.get_pw_poses(), atol=1e-6)


def test_geometry_helpers_match_live_reference():
    """xy_grid / geotrf / inv / depthmap_to_pts3d / depthmap_to_(absolute_)camera_coordinates against what the reference's
    dust3r/utils/geometry.py returns on the same random inputs (CPU; recorded in tests/golden/reference_records.npz), every
    calling convention the two hot paths use."""
    import dust3r_b200.utils.geometry as mine
    gold = reference_records()

    def ref(key, a):
        """The recorded reference output for `key`, after checking that `a` has its type, dtype and shape."""
        b = gold[f'geometry|{key}']
        assert type(a) is (torch.Tensor if str(gold[f'geometry|{key}|type']) == 'torch' else np.ndarray), key
        assert a.dtype == (torch.from_numpy(b).dtype if torch.is_tensor(a) else b.dtype) and tuple(a.shape) == b.shape, key
        return torch.from_numpy(b) if torch.is_tensor(a) else b
    g = torch.Generator().manual_seed(0)
    for i, kw in enumerate((dict(), dict(origin=(2, 3)), dict(homogeneous=True), dict(unsqueeze=0), dict(cat_dim=0))):
        a = mine.xy_grid(7, 5, device='cpu', **kw)
        assert torch.equal(a, ref(f'xy_grid|{i}|cpu', a)), kw
        if 'unsqueeze' not in kw:      # (the reference's numpy branch cannot unsqueeze)
            a = mine.xy_grid(7, 5, **kw)          # device=None -> numpy
            assert np.array_equal(a, ref(f'xy_grid|{i}|none', a)), kw
    T = torch.randn((3, 4, 4), generator=g)
    T[:, 3] = torch.tensor([0., 0, 0, 1])
    P = torch.randn((3, 6, 5, 3), generator=g)
    a = mine.geotrf(T, P)
    assert torch.equal(a, ref('geotrf|batched', a))
    a = mine.geotrf(T[0], P[0])
    assert torch.equal(a, ref('geotrf|single', a))
    K = torch.tensor([[30., 0, 16], [0, 31, 12], [0, 0, 1]])
    a = mine.geotrf(K, P[0], norm=1, ncol=2)
    assert torch.equal(a, ref('geotrf|K', a))
    a = mine.geotrf(T[0].numpy(), P[0].numpy())
    assert np.allclose(a, ref('geotrf|numpy', a))
    a, b = mine.inv(T), mine.inv(T[0].numpy())
    assert torch.equal(a, ref('inv|torch', a)) and np.array_equal(b, ref('inv|numpy', b))
    depth = torch.rand((2, 6, 5), generator=g) + 0.5
    for f, focal in enumerate((torch.rand((2, 1, 6, 5), generator=g) + 20, torch.rand((2, 2, 6, 5), generator=g) + 20)):
        pp = torch.tensor([[2.5, 3.0], [2.0, 3.5]])
        a = mine.depthmap_to_pts3d(depth, focal, pp=pp)
        assert torch.equal(a, ref(f'depthmap_to_pts3d|{f}|pp', a))
        a = mine.depthmap_to_pts3d(depth, focal)
        assert torch.equal(a, ref(f'depthmap_to_pts3d|{f}|nopp', a))
    d = depth[0].numpy()
    d[0, 0] = 0
    xa, ma = mine.depthmap_to_camera_coordinates(d, K.numpy())
    assert np.array_equal(xa, ref('depthmap_to_camera_coordinates|X', xa))
    assert np.array_equal(ma, ref('depthmap_to_camera_coordinates|mask', ma))
    pose = np.eye(4, dtype=np.float32)
    pose[:3, :3] = np.float32([[0, -1, 0], [1, 0, 0], [0, 0, 1]])
    pose[:3, 3] = (1, 2, 3)
    xa, ma = mine.depthmap_to_absolute_camera_coordinates(d, K.numpy(), pose)
    assert np.allclose(xa, ref('depthmap_to_absolute_camera_coordinates|X', xa), atol=1e-6)
    assert np.array_equal(ma, ref('depthmap_to_absolute_camera_coordinates|mask', ma))


def test_stream_work_items_cover_every_slot_once_and_balance():
    """Host-side decomposition of the streaming alignment kernel: every 64-pixel slot of every image belongs to exactly
    one work item, items never cross an image, per-warp lists are contiguous and cost-balanced to within one slot."""
    import numpy as np
    from dust3r_b200.cloud_opt.engine import build_stream_items, SLOT_PX
    rng = np.random.default_rng(0)
    for imshapes, deg in (([(384, 512)] * 8, [7] * 8), ([(24, 32), (20, 36), (14, 44)], [2, 3, 3]), ([(128, 160)] * 50, [49] * 50),
                          ([(8, 16)] * 5, [4, 1, 9, 2, 6])):
        n = len(imshapes)
        areas = [h * w for h, w in imshapes]
        slots = [(a + SLOT_PX - 1) // SLOT_PX for a in areas]
        pix_off = np.concatenate([[0], np.cumsum(areas)]).astype(np.int64)
        ent_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
        ent_obs_off = np.concatenate([[0], np.cumsum(np.repeat(np.array(slots) * SLOT_PX, deg))])[:-1].astype(np.int64)
        items, wptr, grid = build_stream_items(imshapes, pix_off, ent_ptr, ent_obs_off, slots, 3, 8, 296)
        assert len(wptr) == grid * 8 + 1 and wptr[0] == 0 and wptr[-1] == len(items) and np.all(np.diff(wptr) >= 0)
        seen = [np.zeros(s, dtype=int) for s in slots]
        for it in items:
            assert 1 <= it['nslots'] <= 3 and it['slot0'] + it['nslots'] <= slots[it['img']]
            seen[it['img']][it['slot0']:it['slot0'] + it['nslots']] += 1
            p0 = it['slot0'] * SLOT_PX
            H, W = imshapes[it['img']]
            assert it['npx'] == min(it['nslots'] * SLOT_PX, areas[it['img']] - p0) and it['npx'] % 4 == 0
            assert it['v0'] * W + it['u0'] == p0 and it['pix0'] == pix_off[it['img']] + p0
            assert it['obs0'] == ent_obs_off[ent_ptr[it['img']]] + p0 and it['slab_units'] == slots[it['img']] * SLOT_PX
            assert it['e0'] == ent_ptr[it['img']] and it['deg'] == deg[it['img']]
        assert all(np.all(s == 1) for s in seen)
        # items of one warp are consecutive slots of the global sequence
        glob = np.concatenate([[0], np.cumsum(slots)])
        cost = []
        for w in range(grid * 8):
            its = items[wptr[w]:wptr[w + 1]]
            pos = [glob[i['img']] + i['slot0'] for i in its]
            assert all(pos[k + 1] == pos[k] + its[k]['nslots'] for k in range(len(its) - 1))
            cost.append(sum(int(i['nslots']) * (int(i['deg']) + 3) for i in its))
        busy = [c for c in cost if c > 0]
        assert max(busy) - min(busy) <= 2 * (max(deg) + 3), (max(busy), min(busy))


def test_find_reciprocal_matches_host_path_matches_live_reference():
    """utils/geometry.py:345-361 (scipy cKDTree on the CPU, like the reference; its result recorded in
    tests/golden/reference_records.npz); the CUDA path is checked against this one in tests/test_scene_ops_gpu.py."""
    from dust3r_b200.utils.geometry import find_reciprocal_matches as mine
    gold = reference_records()
    rng = np.random.default_rng(0)
    P1 = rng.standard_normal((700, 3)).astype(np.float32)
    P2 = np.concatenate((P1[:400] + 0.01 * rng.standard_normal((400, 3)).astype(np.float32), rng.standard_normal((150, 3)).astype(np.float32)))
    assert digest(P1) + digest(P2) == str(gold['reciprocal|inputs']), 'inputs differ from the recorded ones'
    a, b = [gold[f'reciprocal|{k}'] for k in range(3)], mine(P1, P2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and int(a[2]) == int(b[2]) > 300


def test_load_model_and_from_pretrained_on_a_reference_format_checkpoint(tmp_path):
    """dust3r/model.py:27-43, 76-85: a checkpoint is {'args': Namespace(model="AsymmetricCroCo3DStereo(...)"), 'model': state
    dict}; load_model rebuilds the network from the constructor string (ManyAR_PatchEmbed -> PatchEmbedDust3R,
    landscape_only forced to False) and loads the weights; from_pretrained(path) of an existing file does the same.  No real
    checkpoint is available offline: a small synthetic one is written in that format; the state dict the reference's own
    load_model reads back from it is recorded in tests/golden/reference_records.npz (one digest per tensor)."""
    import argparse
    from dust3r_b200.config import ModelConfig
    from dust3r_b200.model import AsymmetricCroCo3DStereo, load_model
    from dust3r_b200.utils.synth import synth_state_dict
    cfg = ModelConfig(img_size=(96, 96), enc_embed_dim=192, enc_depth=3, enc_num_heads=3, dec_embed_dim=128, dec_depth=2,
                      dec_num_heads=2, head_type='linear', landscape_only=False)
    sd = synth_state_dict(cfg, seed=4)
    ctor = ("AsymmetricCroCo3DStereo(pos_embed='RoPE100', patch_embed_cls='ManyAR_PatchEmbed', img_size=(96, 96), head_type='linear', "
            "output_mode='pts3d', depth_mode=('exp', -inf, inf), conf_mode=('exp', 1, inf), enc_embed_dim=192, enc_depth=3, "
            "enc_num_heads=3, dec_embed_dim=128, dec_depth=2, dec_num_heads=2)")
    path = str(tmp_path / 'synthetic_checkpoint.pth')
    # released checkpoints predate dec_blocks2 in some cases: drop them so that the duplication rule (model.py:91-98) is exercised
    stored = {k: v for k, v in sd.items() if not k.startswith('dec_blocks2')}
    torch.save({'args': argparse.Namespace(model=ctor), 'model': stored}, path)
    net = load_model(path, 'cpu', verbose=False)
    assert isinstance(net, AsymmetricCroCo3DStereo) and net.landscape_only is False
    got = net.state_dict()
    assert set(got) == set(sd)
    for k, v in sd.items():
        src = sd[k.replace('dec_blocks2', 'dec_blocks')] if k.startswith('dec_blocks2') else v
        assert torch.equal(got[k], src), k
    net2 = AsymmetricCroCo3DStereo.from_pretrained(path)
    assert all(torch.equal(a, b) for a, b in zip(net2.state_dict().values(), got.values()))
    gold = reference_records()
    assert sorted(got) == gold['load_model|keys'].tolist()
    assert [digest(got[k]) for k in sorted(got)] == gold['load_model|digests'].tolist()


@pytest.mark.parametrize('imshapes,n_edges', [([(384, 512)] * 8, 28), ([(32, 48), (48, 32), (16, 64), (64, 64)], 5), ([(8, 8), (24, 40)], 1)])
def test_stream_items_partition_every_image_exactly_once(imshapes, n_edges):
    """Work-item tables of the streaming alignment kernel (engine.build_stream_items, numpy): every 64-pixel slot of every image
    is covered exactly once, in order; no item crosses an image or a warp boundary or exceeds 3 slots; pixel / observation
    offsets follow from the slot index; the reversed traversal built on top of it visits the same items backwards."""
    from dust3r_b200.cloud_opt.engine import build_stream_items, SLOT_PX
    n = len(imshapes)
    edges = [(i, j) for i in range(n) for j in range(i)][:n_edges]
    areas = [h * w for h, w in imshapes]
    pix_off = np.zeros(n + 1, dtype=np.int64)
    pix_off[1:] = np.cumsum(areas)
    ent = [[] for _ in range(n)]
    for e, (i, j) in enumerate(edges):
        ent[i].append(e)
        ent[j].append(e)
    ent_ptr = np.zeros(n + 1, dtype=np.int32)
    ent_ptr[1:] = np.cumsum([len(l) for l in ent])
    slots = [(a + SLOT_PX - 1) // SLOT_PX for a in areas]
    ent_obs_off = np.zeros(2 * len(edges), dtype=np.int64)
    off = k = 0
    for i in range(n):
        for _ in ent[i]:
            ent_obs_off[k] = off
            off += slots[i] * SLOT_PX
            k += 1
    items, warp_ptr, grid = build_stream_items(imshapes, pix_off, ent_ptr, ent_obs_off, slots, 3, 8, 296)
    assert warp_ptr[0] == 0 and warp_ptr[-1] == len(items) and len(warp_ptr) == grid * 8 + 1 and np.all(np.diff(warp_ptr) >= 0)
    covered = {i: 0 for i in range(n)}
    for it in items:
        i = int(it['img'])
        assert it['slot0'] == covered[i] and 1 <= it['nslots'] <= 3           # in order, gap-free
        covered[i] += int(it['nslots'])
        p0 = int(it['slot0']) * SLOT_PX
        H, W = imshapes[i]
        assert it['npx'] == min(int(it['nslots']) * SLOT_PX, areas[i] - p0) and it['npx'] % 4 == 0
        assert it['pix0'] == pix_off[i] + p0 and it['W'] == W and it['u0'] == p0 % W and it['v0'] == p0 // W
        assert it['e0'] == ent_ptr[i] and it['deg'] == ent_ptr[i + 1] - ent_ptr[i] and it['slab_units'] == slots[i] * SLOT_PX
        if it['deg'] > 0:
            assert it['obs0'] == ent_obs_off[ent_ptr[i]] + p0
    assert all(covered[i] == slots[i] for i in range(n))
    # a warp's run never mixes images inside one item (checked above) and is contiguous in the global slot order
    starts = np.asarray([np.cumsum([0] + slots)[int(it['img'])] + int(it['slot0']) for it in items])
    assert np.all(np.diff(starts) > 0)
