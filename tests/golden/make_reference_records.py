"""Records what the UNMODIFIED reference returns for the CPU-side comparisons of the suite (host API of cloud_opt, geometry
helpers, init='mst', PairViewer, ModularPointCloudOptimizer presets, is_symmetrized, load_model, load_images and one small
forward) into tests/golden/reference_records.npz, so that those tests run without the reference.

    python tests/golden/make_reference_records.py <reference checkout>

Every section below replays the reference side of one test, on the same synthetic inputs in the same order of random draws.
Large outputs that a test compares bit for bit are stored as sha256 digests (digest(): dtype, shape and bytes); outputs
compared with a tolerance are stored as values, the two largest (pointmaps of the symmetrised forward and of PairViewer) at a
fixed, seeded quarter of the pixel positions, which are stored with them (keeps the fixture small).
"""
import argparse
import copy
import hashlib
import itertools
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, 'reference_records.npz')
inf = float('inf')


def digest(a):
    """sha256 over dtype, shape and bytes of an array or tensor: equal digests <=> torch.equal / np.array_equal with equal
    dtype and shape."""
    if torch.is_tensor(a):
        a = a.detach().cpu().contiguous().numpy()
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f'{a.dtype.str}|{a.shape}|'.encode())
    h.update(a.tobytes())
    return h.hexdigest()


def _np(t):
    return t.detach().cpu().numpy().copy() if torch.is_tensor(t) else np.asarray(t).copy()


def pixel_sample(n_px, seed=0):
    """Sorted indices of a fixed quarter of n_px flattened pixel positions."""
    return np.sort(np.random.default_rng(seed).choice(n_px, n_px // 4, replace=False)).astype(np.int64)


def _edges_sym(n):
    e = [(i, j) for i in range(n) for j in range(i)]
    return e + [(j, i) for i, j in e]


def optimizer_init_draws(res):
    """tests/test_host_logic.py::test_optimizer_init_matches_reference_draws"""
    from dust3r.cloud_opt import global_aligner, GlobalAlignerMode
    from dust3r_b200.utils.synth import synth_pair_predictions
    n, H, W = 3, 16, 32
    out = synth_pair_predictions(n, [(i, j) for i in range(n) for j in range(i)], H, W, seed=2)
    torch.manual_seed(123)
    ref = global_aligner(copy.deepcopy(out), 'cpu', mode=GlobalAlignerMode.PointCloudOptimizer, verbose=False)
    for k in ('pw_poses', 'im_depthmaps', 'im_poses', 'im_focals', 'im_pp'):
        res[f'init_draws|{k}'] = _np(getattr(ref, k).data)
    for i, p in enumerate(ref.get_pts3d()):
        res[f'init_draws|pts3d|{i}'] = _np(p)
    res['init_draws|get_pw_poses'] = _np(ref.get_pw_poses())


def geometry_helpers(res):
    """tests/test_host_logic.py::test_geometry_helpers_match_live_reference"""
    import dust3r.utils.geometry as ref
    g = torch.Generator().manual_seed(0)

    def put(key, a):
        res[f'geometry|{key}'] = _np(a)
        res[f'geometry|{key}|type'] = np.str_('torch' if torch.is_tensor(a) else 'numpy')
    for i, kw in enumerate((dict(), dict(origin=(2, 3)), dict(homogeneous=True), dict(unsqueeze=0), dict(cat_dim=0))):
        put(f'xy_grid|{i}|cpu', ref.xy_grid(7, 5, device='cpu', **kw))
        if 'unsqueeze' not in kw:
            put(f'xy_grid|{i}|none', ref.xy_grid(7, 5, **kw))
    T = torch.randn((3, 4, 4), generator=g)
    T[:, 3] = torch.tensor([0., 0, 0, 1])
    P = torch.randn((3, 6, 5, 3), generator=g)
    put('geotrf|batched', ref.geotrf(T, P))
    put('geotrf|single', ref.geotrf(T[0], P[0]))
    K = torch.tensor([[30., 0, 16], [0, 31, 12], [0, 0, 1]])
    put('geotrf|K', ref.geotrf(K, P[0], norm=1, ncol=2))
    put('geotrf|numpy', ref.geotrf(T[0].numpy(), P[0].numpy()))
    put('inv|torch', ref.inv(T))
    put('inv|numpy', ref.inv(T[0].numpy()))
    depth = torch.rand((2, 6, 5), generator=g) + 0.5
    for f, focal in enumerate((torch.rand((2, 1, 6, 5), generator=g) + 20, torch.rand((2, 2, 6, 5), generator=g) + 20)):
        pp = torch.tensor([[2.5, 3.0], [2.0, 3.5]])
        put(f'depthmap_to_pts3d|{f}|pp', ref.depthmap_to_pts3d(depth, focal, pp=pp))
        put(f'depthmap_to_pts3d|{f}|nopp', ref.depthmap_to_pts3d(depth, focal))
    d = depth[0].numpy()
    d[0, 0] = 0
    x, m = ref.depthmap_to_camera_coordinates(d, K.numpy())
    put('depthmap_to_camera_coordinates|X', x)
    put('depthmap_to_camera_coordinates|mask', m)
    pose = np.eye(4, dtype=np.float32)
    pose[:3, :3] = np.float32([[0, -1, 0], [1, 0, 0], [0, 0, 1]])
    pose[:3, 3] = (1, 2, 3)
    x, m = ref.depthmap_to_absolute_camera_coordinates(d, K.numpy(), pose)
    put('depthmap_to_absolute_camera_coordinates|X', x)
    put('depthmap_to_absolute_camera_coordinates|mask', m)


def reciprocal_matches(res):
    """tests/test_host_logic.py::test_find_reciprocal_matches_host_path_matches_live_reference"""
    from dust3r.utils.geometry import find_reciprocal_matches
    rng = np.random.default_rng(0)
    P1 = rng.standard_normal((700, 3)).astype(np.float32)
    P2 = np.concatenate((P1[:400] + 0.01 * rng.standard_normal((400, 3)).astype(np.float32), rng.standard_normal((150, 3)).astype(np.float32)))
    a = find_reciprocal_matches(P1, P2)
    res['reciprocal|inputs'] = np.str_(digest(P1) + digest(P2))
    for k in range(3):
        res[f'reciprocal|{k}'] = np.asarray(a[k])


def load_model_checkpoint(res):
    """tests/test_host_logic.py::test_load_model_and_from_pretrained_on_a_reference_format_checkpoint: the same synthetic
    checkpoint, read back by the reference's load_model; its state dict stored as key -> digest."""
    from dust3r.model import load_model
    from dust3r_b200.config import ModelConfig
    from dust3r_b200.utils.synth import synth_state_dict
    cfg = ModelConfig(img_size=(96, 96), enc_embed_dim=192, enc_depth=3, enc_num_heads=3, dec_embed_dim=128, dec_depth=2,
                      dec_num_heads=2, head_type='linear', landscape_only=False)
    sd = synth_state_dict(cfg, seed=4)
    ctor = ("AsymmetricCroCo3DStereo(pos_embed='RoPE100', patch_embed_cls='ManyAR_PatchEmbed', img_size=(96, 96), head_type='linear', "
            "output_mode='pts3d', depth_mode=('exp', -inf, inf), conf_mode=('exp', 1, inf), enc_embed_dim=192, enc_depth=3, "
            "enc_num_heads=3, dec_embed_dim=128, dec_depth=2, dec_num_heads=2)")
    stored = {k: v for k, v in sd.items() if not k.startswith('dec_blocks2')}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, 'synthetic_checkpoint.pth')
        torch.save({'args': argparse.Namespace(model=ctor), 'model': stored}, path)
        with torch.serialization.safe_globals([argparse.Namespace]):
            rsd = load_model(path, 'cpu', verbose=False).state_dict()
    keys = sorted(rsd)
    res['load_model|keys'] = np.array(keys)
    res['load_model|digests'] = np.array([digest(rsd[k]) for k in keys])


def mst_init(res):
    """tests/test_init_poses.py::test_mst_init_matches_reference"""
    import cv2
    from dust3r.cloud_opt import global_aligner
    import dust3r.cloud_opt.init_im_poses as init_im_poses
    from dust3r_b200.utils.synth import synth_consistent_scene
    out, cams, f = synth_consistent_scene(4, _edges_sym(4), 24, 32, seed=2, noise=0.005)
    torch.manual_seed(3)
    cv2.setRNGSeed(0)
    ref = global_aligner(copy.deepcopy(out), 'cpu', verbose=False)
    ref.verbose = False
    init_im_poses.init_minimum_spanning_tree(ref, niter_PnP=10)
    for k in ('pw_poses', 'im_poses', 'im_focals', 'im_depthmaps'):
        res[f'mst|{k}'] = _np(getattr(ref, k).data)


def pair_viewer(res):
    """tests/test_init_poses.py::test_pair_viewer_matches_live_reference"""
    import cv2
    from dust3r.cloud_opt import global_aligner, GlobalAlignerMode
    from dust3r_b200.utils.synth import synth_consistent_scene
    out, cams, f = synth_consistent_scene(2, [(0, 1), (1, 0)], 48, 64, seed=3, noise=0.002)
    cv2.setRNGSeed(0)
    b = global_aligner(copy.deepcopy(out), 'cpu', mode=GlobalAlignerMode.PairViewer, verbose=False)
    for get in ('get_focals', 'get_im_poses', 'get_principal_points', 'get_intrinsics'):
        res[f'pair_viewer|{get}'] = _np(getattr(b, get)())
    for get in ('get_depthmaps', 'get_masks'):
        for i, x in enumerate(getattr(b, get)()):
            res[f'pair_viewer|{get}|{i}'] = _np(x)
    px = res['pair_viewer|px'] = pixel_sample(48 * 64)
    for i, x in enumerate(b.get_pts3d()):
        res[f'pair_viewer|get_pts3d|{i}'] = _np(x).reshape(-1, 3)[px]


def is_symmetrized(res):
    """tests/test_init_poses.py::test_is_symmetrized_quirks_match_live_reference: 1 / 0 / -1 (IndexError) for every couple of
    instance lists of length <= 5 over 'ab', in itertools.product order."""
    from dust3r.utils.misc import is_symmetrized as fn
    outcomes = []
    for n in range(1, 6):
        for a in itertools.product('ab', repeat=n):
            for b in itertools.product('ab', repeat=n):
                try:
                    outcomes.append(int(bool(fn(dict(instance=list(a)), dict(instance=list(b))))))
                except IndexError:
                    outcomes.append(-1)
    res['is_symmetrized|outcomes'] = np.int8(outcomes)


def modular_presets(res):
    """tests/test_init_poses.py::test_modular_optimizer_presets_match_live_reference (both fx_and_fy)"""
    from dust3r.cloud_opt import global_aligner, GlobalAlignerMode
    from dust3r_b200.utils.synth import synth_pair_predictions
    n, H, W = 4, 24, 32
    out = synth_pair_predictions(n, [(i, j) for i in range(n) for j in range(n) if i != j], H, W, seed=2)
    for fx_and_fy in (False, True):
        torch.manual_seed(0)
        b = global_aligner(copy.deepcopy(out), 'cpu', mode=GlobalAlignerMode.ModularPointCloudOptimizer, verbose=False,
                           fx_and_fy=fx_and_fy, optimize_pp=True)
        Ks = [torch.tensor([[30. + i, 0, 15 + i], [0, 32. + i, 11 - i], [0, 0, 1.]]) for i in range(2)]
        poses = [torch.eye(4), torch.tensor([[0., -1, 0, 1], [1, 0, 0, 2], [0, 0, 1, 3], [0, 0, 0, 1]])]
        b.preset_intrinsics(Ks, msk=[1, 3])
        b.preset_pose(poses, pose_msk=torch.tensor([True, False, True, False]))
        b.preset_focal([55.0], msk=0)
        b.preset_principal_point([torch.tensor([14., 13.])], msk=np.array([2]))
        p = f'modular|{int(fx_and_fy)}'
        res[f'{p}|norm_pw_scale'] = np.bool_(b.norm_pw_scale)
        for name in ('im_poses', 'im_pp', 'im_focals'):
            res[f'{p}|requires_grad|{name}'] = np.bool_([q.requires_grad for q in getattr(b, name)])
        for get in ('get_focals', 'get_principal_points', 'get_intrinsics', 'get_im_poses'):
            res[f'{p}|{get}'] = _np(getattr(b, get)())
        res[f'{p}|get_pts3d'] = np.array([digest(x) for x in b.get_pts3d()])
        res[f'{p}|get_depthmaps'] = np.array([digest(x) for x in b.get_depthmaps()])


def forward_symmetrised_batch(res):
    """tests/test_oracle.py::test_forward_oracle_bit_matches_live_reference: a symmetrised batch of two pairs (half-encoder
    path of the reference)."""
    from dust3r.model import AsymmetricCroCo3DStereo
    from dust3r_b200.config import ModelConfig
    from dust3r_b200.utils.synth import synth_state_dict, synth_images
    cfg = ModelConfig(img_size=(64, 64), enc_embed_dim=128, enc_depth=2, enc_num_heads=2, dec_embed_dim=64,
                      dec_depth=10, dec_num_heads=1, head_type='dpt', landscape_only=False)
    m = AsymmetricCroCo3DStereo(
        pos_embed=cfg.pos_embed, patch_embed_cls='PatchEmbedDust3R', img_size=cfg.img_size, head_type=cfg.head_type,
        output_mode='pts3d', depth_mode=cfg.depth_mode, conf_mode=cfg.conf_mode, enc_embed_dim=cfg.enc_embed_dim,
        enc_depth=cfg.enc_depth, enc_num_heads=cfg.enc_num_heads, dec_embed_dim=cfg.dec_embed_dim,
        dec_depth=cfg.dec_depth, dec_num_heads=cfg.dec_num_heads, landscape_only=cfg.landscape_only).eval()
    sd = synth_state_dict(cfg, seed=21)
    m.load_state_dict(sd, strict=True)
    imgs = synth_images(4, 48, 64, seed=9)
    img1 = torch.cat([imgs[0]['img'], imgs[1]['img']])
    img2 = torch.cat([imgs[1]['img'], imgs[0]['img']])
    ts = torch.tensor([[48, 64]] * 2)
    with torch.no_grad():
        r1, r2 = m(dict(img=img1, true_shape=ts, instance=['0', '1']), dict(img=img2, true_shape=ts, instance=['1', '0']))
    res['forward_sym|inputs'] = np.str_(digest(img1) + digest(img2))
    px = res['forward_sym|px'] = pixel_sample(48 * 64)
    for key, t in (('pts3d', r1['pts3d']), ('conf1', r1['conf']), ('pts3d_in_other_view', r2['pts3d_in_other_view']),
                   ('conf2', r2['conf'])):
        res[f'forward_sym|{key}'] = _np(t).reshape(2, 48 * 64, -1)[:, px]


LOAD_IMAGES_CASES = [  # (H, W, size, square_ok): tests/test_image_preprocess.py::CASES, photo seed 10 + index
    (150, 200, 128, False), (200, 150, 128, False), (130, 130, 128, False), (130, 130, 128, True), (37, 53, 224, False),
    (300, 170, 224, False), (480, 640, 512, False), (640, 480, 512, False), (90, 70, 160, False), (384, 512, 512, False),
    (97, 1003, 512, False), (601, 397, 224, False), (224, 224, 224, False),
]


def load_images_files(res):
    """tests/test_image_preprocess.py::test_oracle_and_host_port_equal_live_reference_load_images (one PNG per case) and
    ::test_load_images_folder_threads_keep_the_sequential_contract (a folder of PNG / JPEG files and one text file)."""
    import PIL.Image
    from dust3r.utils.image import load_images
    from dust3r_b200.utils.synth import synth_photo
    with tempfile.TemporaryDirectory() as tmp:
        for k, (h, w, size, sq) in enumerate(LOAD_IMAGES_CASES):
            photo = synth_photo(h, w, seed=10 + k)
            path = os.path.join(tmp, f'{k}.png')
            PIL.Image.fromarray(photo).save(path)
            v = load_images([path], size=size, square_ok=sq, verbose=False)[0]
            res[f'load_images|{k}|photo'] = np.str_(digest(photo))
            res[f'load_images|{k}|img'] = np.str_(digest(v['img']))
            res[f'load_images|{k}|true_shape'] = np.asarray(v['true_shape'])
            res[f'load_images|{k}|idx'] = np.int64(v['idx'])
            res[f'load_images|{k}|instance'] = np.str_(v['instance'])
    shapes = [(90, 120), (120, 90), (100, 100), (64, 200), (33, 47), (150, 151), (80, 81)]
    with tempfile.TemporaryDirectory() as tmp:
        for k, (h, w) in enumerate(shapes):
            PIL.Image.fromarray(synth_photo(h, w, seed=50 + k)).save(os.path.join(tmp, f'im{k:02d}.{"png" if k % 2 else "jpg"}'))
        open(os.path.join(tmp, 'readme.txt'), 'w').write('not an image')
        views = load_images(tmp, size=64, verbose=False)
    res['load_images_folder|img'] = np.array([digest(v['img']) for v in views])
    res['load_images_folder|true_shape'] = np.concatenate([np.asarray(v['true_shape']) for v in views])
    res['load_images_folder|instance'] = np.array([v['instance'] for v in views])


SECTIONS = [optimizer_init_draws, geometry_helpers, reciprocal_matches, load_model_checkpoint, mst_init, pair_viewer,
            is_symmetrized, modular_presets, forward_symmetrised_batch, load_images_files]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('reference', help='checkout of the reference project (the directory that holds dust3r/)')
    args = ap.parse_args()
    if not os.path.isdir(os.path.join(args.reference, 'dust3r')):
        raise SystemExit(f'{args.reference}: no dust3r/ package there')
    # `roma` is not installable offline: the reference's cloud_opt runs on the local restatement of its three entry points
    sys.path[:0] = [os.path.abspath(args.reference), os.path.join(ROOT, 'oracle', 'roma_stub'), ROOT]
    res = {}
    for section in SECTIONS:
        section(res)
        print(section.__name__, 'done')
    np.savez_compressed(OUT, **res)
    print('wrote', OUT, os.path.getsize(OUT), 'bytes')


if __name__ == '__main__':
    main()
