"""Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on CPU fp32.

    python tests/golden/make_golden.py            # in the build container (reference mounted)

Forward goldens come from the pure reference.  Alignment goldens are "reference cloud_opt + local roma
restatement" (oracle/roma_stub) because `roma` is not installable offline (SURVEY §8c).
Inputs/weights are regenerated from dust3r_b200.utils.synth by the tests (deterministic), so the
fixtures only hold the reference's OUTPUTS plus input checksums.
"""
import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle', 'roma_stub'))
sys.path.insert(0, '/root/reference')
sys.path.insert(0, ROOT)

from dust3r_b200.config import ModelConfig, vitl_512_dpt, vitl_224_linear  # noqa: E402
from dust3r_b200.utils.synth import synth_state_dict, synth_images, synth_pair_predictions, many_ar_inputs  # noqa: E402

inf = float('inf')


def ref_model(cfg, patch_embed_cls='PatchEmbedDust3R'):
    from dust3r.model import AsymmetricCroCo3DStereo
    m = AsymmetricCroCo3DStereo(
        pos_embed=cfg.pos_embed, patch_embed_cls=patch_embed_cls, img_size=cfg.img_size, head_type=cfg.head_type,
        output_mode='pts3d', depth_mode=cfg.depth_mode, conf_mode=cfg.conf_mode, enc_embed_dim=cfg.enc_embed_dim,
        enc_depth=cfg.enc_depth, enc_num_heads=cfg.enc_num_heads, dec_embed_dim=cfg.dec_embed_dim,
        dec_depth=cfg.dec_depth, dec_num_heads=cfg.dec_num_heads, landscape_only=cfg.landscape_only).eval()
    return m


SMALL = dict(
    small_dpt=(ModelConfig(img_size=(96, 96), enc_embed_dim=128, enc_depth=2, enc_num_heads=2, dec_embed_dim=128,
                           dec_depth=12, dec_num_heads=2, head_type='dpt', landscape_only=False), 64, 96),
    small_linear=(ModelConfig(img_size=(96, 96), enc_embed_dim=192, enc_depth=3, enc_num_heads=3, dec_embed_dim=128,
                              dec_depth=2, dec_num_heads=2, head_type='linear', landscape_only=False), 80, 64),
)


def many_ar_golden():
    """landscape_only=True + ManyAR_PatchEmbed (the training-time configuration): transposed portrait items in a landscape
    batch -> ManyAR_PatchEmbed.forward (patch_embed.py:42-70) and transpose_to_landscape.wrapper_yes (utils/misc.py:66-95)."""
    for name in ('small_linear', 'small_dpt'):
        cfg0, H, W = SMALL[name]
        H, W = min(H, W), max(H, W)
        cfg = copy.deepcopy(cfg0)
        cfg.landscape_only = True
        m = ref_model(cfg, patch_embed_cls='ManyAR_PatchEmbed')
        sd = synth_state_dict(cfg, seed=11)
        m.load_state_dict(sd, strict=True)
        v1, v2 = many_ar_inputs(H, W)
        with torch.no_grad():
            r1, r2 = m(v1, v2)
        np.savez_compressed(os.path.join(HERE, f'forward_{name}_manyar.npz'), H=H, W=W,
                            pts3d=r1['pts3d'].numpy(), conf1=r1['conf'].numpy(),
                            pts3d_in_other_view=r2['pts3d_in_other_view'].numpy(), conf2=r2['conf'].numpy())
        print('wrote many-AR', name, r1['pts3d'].shape)


def forward_goldens():
    from dust3r.inference import inference
    from dust3r.image_pairs import make_pairs
    for name, (cfg, H, W) in SMALL.items():
        torch.manual_seed(0)
        m = ref_model(cfg)
        sd = synth_state_dict(cfg, seed=11)
        m.load_state_dict(sd, strict=True)
        imgs = synth_images(3, H, W, seed=5)
        pairs = make_pairs(imgs, scene_graph='complete', prefilter=None, symmetrize=True)   # 6 pairs
        out = inference(pairs, m, 'cpu', batch_size=4, verbose=False)
        np.savez_compressed(os.path.join(HERE, f'forward_{name}.npz'),
                            pts3d=out['pred1']['pts3d'].numpy(), conf1=out['pred1']['conf'].numpy(),
                            pts3d_in_other_view=out['pred2']['pts3d_in_other_view'].numpy(),
                            conf2=out['pred2']['conf'].numpy(),
                            idx1=np.int64(out['view1']['idx']), idx2=np.int64(out['view2']['idx']),
                            img_sum=np.float64([float(i['img'].double().sum()) for i in imgs]))
        print('wrote', name, out['pred1']['pts3d'].shape)

    many_ar_golden()

    # the two published architectures, one 1-pair batch each, strided sample of the outputs
    for name, cfg, H, W, stride in (('vitl_512_dpt', vitl_512_dpt(), 384, 512, 8), ('vitl_224_linear', vitl_224_linear(), 224, 224, 4)):
        m = ref_model(cfg)
        sd = synth_state_dict(cfg, seed=0)
        m.load_state_dict(sd, strict=True)
        imgs = synth_images(2, H, W, seed=3)
        out = inference([(imgs[0], imgs[1])], m, 'cpu', batch_size=1, verbose=False)
        s = stride
        np.savez_compressed(os.path.join(HERE, f'forward_{name}.npz'), stride=s,
                            pts3d=out['pred1']['pts3d'][:, ::s, ::s].numpy(), conf1=out['pred1']['conf'][:, ::s, ::s].numpy(),
                            pts3d_in_other_view=out['pred2']['pts3d_in_other_view'][:, ::s, ::s].numpy(),
                            conf2=out['pred2']['conf'][:, ::s, ::s].numpy(),
                            mean_abs=np.float64([out['pred1']['pts3d'].abs().mean(), out['pred1']['conf'].mean(),
                                                 out['pred2']['pts3d_in_other_view'].abs().mean(), out['pred2']['conf'].mean()]))
        print('wrote', name)


ODD_GRID_SIZES = [(48, 80), (80, 48)]   # small_dpt at 3x5 and 5x3 tokens: odd grid width and height in the DPT head


def forward_odd_grid_goldens():
    """small_dpt on token grids with an odd width or height, same flow as forward_goldens: the stride-2 conv of
    act_postprocess 3 rounds the grid up and refinenet4's x2 output is cropped back to the grid (heads/dpt_head.py:57)."""
    from dust3r.inference import inference
    from dust3r.image_pairs import make_pairs
    cfg = SMALL['small_dpt'][0]
    for H, W in ODD_GRID_SIZES:
        torch.manual_seed(0)
        m = ref_model(cfg)
        sd = synth_state_dict(cfg, seed=11)
        m.load_state_dict(sd, strict=True)
        imgs = synth_images(3, H, W, seed=5)
        pairs = make_pairs(imgs, scene_graph='complete', prefilter=None, symmetrize=True)
        out = inference(pairs, m, 'cpu', batch_size=4, verbose=False)
        np.savez_compressed(os.path.join(HERE, f'forward_small_dpt_{H}x{W}.npz'),
                            pts3d=out['pred1']['pts3d'].numpy(), conf1=out['pred1']['conf'].numpy(),
                            pts3d_in_other_view=out['pred2']['pts3d_in_other_view'].numpy(),
                            conf2=out['pred2']['conf'].numpy(),
                            idx1=np.int64(out['view1']['idx']), idx2=np.int64(out['view2']['idx']),
                            img_sum=np.float64([float(i['img'].double().sum()) for i in imgs]))
        print('wrote odd grid', (H, W), out['pred1']['pts3d'].shape)


def forward_mixed_goldens():
    from dust3r.inference import inference
    from dust3r.image_pairs import make_pairs
    # mixed image sizes: three images of different sizes, all 6 ordered pairs -> the reference forces batch size 1,
    # returns lists, and encodes the two views of every pair separately (model.py:147-151)
    for name, (cfg, H, W) in SMALL.items():
        torch.manual_seed(0)
        m = ref_model(cfg)
        sd = synth_state_dict(cfg, seed=11)
        m.load_state_dict(sd, strict=True)
        sizes = [(H, W), (H - 16, W), (H, W - 32)]
        imgs = [dict(synth_images(1, h, w, seed=20 + k)[0], idx=k, instance=str(k)) for k, (h, w) in enumerate(sizes)]
        pairs = make_pairs(imgs, scene_graph='complete', prefilter=None, symmetrize=True)
        out = inference(pairs, m, 'cpu', batch_size=4, verbose=False)
        res = dict(idx1=np.int64(out['view1']['idx']), idx2=np.int64(out['view2']['idx']))
        for k in range(len(pairs)):
            res[f'pts3d_{k}'] = out['pred1']['pts3d'][k].numpy()
            res[f'conf1_{k}'] = out['pred1']['conf'][k].numpy()
            res[f'pts3d_in_other_view_{k}'] = out['pred2']['pts3d_in_other_view'][k].numpy()
            res[f'conf2_{k}'] = out['pred2']['conf'][k].numpy()
        np.savez_compressed(os.path.join(HERE, f'forward_{name}_mixed.npz'), **res)
        print('wrote mixed', name, [tuple(out['pred1']['pts3d'][k].shape) for k in range(len(pairs))])


def pair_goldens():
    from dust3r.image_pairs import make_pairs
    res = {}
    for n in (2, 3, 8, 50):
        imgs = [dict(idx=i, instance=str(i)) for i in range(n)]
        for sg in ('complete', 'swin-3', 'swin-5-noncyclic', 'logwin-3', 'logwin-4-noncyclic', 'oneref-0', 'oneref-1'):
            for sym in (True, False):
                for pf in (None, 'seq3', 'cyc3'):
                    pairs = make_pairs(imgs, scene_graph=sg, prefilter=pf, symmetrize=sym)
                    res[f'{n}|{sg}|{int(sym)}|{pf}'] = np.int32([(a['idx'], b['idx']) for a, b in pairs]).reshape(-1, 2)
    np.savez_compressed(os.path.join(HERE, 'make_pairs.npz'), **res)
    print('wrote make_pairs', len(res))


def align_goldens():
    from dust3r.cloud_opt import global_aligner, GlobalAlignerMode
    from dust3r.cloud_opt.base_opt import global_alignment_iter
    from oracle.align_oracle import AlignProblem, init_params
    n, H, W = 4, 24, 32
    edges = [(i, j) for i in range(n) for j in range(i)]
    edges = edges + [(j, i) for i, j in edges]
    res = {}
    for mode, variant in ((GlobalAlignerMode.PointCloudOptimizer, 'stacked'), (GlobalAlignerMode.ModularPointCloudOptimizer, 'per_edge')):
        for dist in ('l1', 'l2'):
            for schedule in ('cosine', 'linear'):
                out = synth_pair_predictions(n, edges, H, W, seed=1)
                net = global_aligner(copy.deepcopy(out), 'cpu', mode=mode, verbose=False, dist=dist)
                prob = AlignProblem.from_output(out, dist=dist, variant=variant)
                P0 = init_params(prob, seed=5)
                with torch.no_grad():
                    if variant == 'stacked':
                        net.im_depthmaps.data[:] = torch.stack(P0['im_depthmaps'])
                        net.im_poses.data[:] = P0['im_poses']
                        net.im_focals.data[:] = P0['im_focals']
                    else:
                        for i in range(n):
                            net.im_depthmaps[i].data[:] = P0['im_depthmaps'][i].view(H, W)
                            net.im_poses[i].data[:] = P0['im_poses'][i]
                            net.im_focals[i].data[:] = P0['im_focals'][i]
                    net.pw_poses.data[:] = P0['pw_poses']
                niter = 60
                params = [p for p in net.parameters() if p.requires_grad]
                opt = torch.optim.Adam(params, lr=0.01, betas=(0.9, 0.9))
                losses = [global_alignment_iter(net, it, niter, 0.01, 1e-6, opt, schedule)[0] for it in range(niter)]
                key = f'{variant}|{dist}|{schedule}'
                res[key + '|loss'] = np.float32(losses)
                if variant == 'stacked':
                    res[key + '|depth'] = net.im_depthmaps.detach().numpy()
                    res[key + '|poses'] = net.im_poses.detach().numpy()
                    res[key + '|focals'] = net.im_focals.detach().numpy()
                else:
                    res[key + '|depth'] = torch.stack([d.detach().reshape(-1) for d in net.im_depthmaps]).numpy()
                    res[key + '|poses'] = torch.stack([d.detach() for d in net.im_poses]).numpy()
                    res[key + '|focals'] = torch.stack([d.detach() for d in net.im_focals]).numpy()
                res[key + '|pw'] = net.pw_poses.detach().numpy()
                print(key, losses[0], losses[-1])
    np.savez_compressed(os.path.join(HERE, 'align_n4.npz'), **res)


IMAGE_CASES = [  # (H, W, seed, size, square_ok): shrinking (Lanczos) and enlarging (bicubic), both orientations, squares
    (150, 200, 1, 128, False), (200, 150, 2, 128, False), (130, 130, 3, 128, False), (130, 130, 3, 128, True),
    (37, 53, 4, 224, False), (300, 170, 5, 224, False), (200, 300, 6, 256, False), (90, 70, 7, 160, False),
]


def image_goldens():
    """load_images of the UNMODIFIED reference (PIL resize / crop + torchvision ImgNorm) on synthetic photographs written
    as PNG files.  The fixture holds the decoded inputs and the reference's outputs; an output has only 256 possible
    values per element ((v / 255 - 0.5) / 0.5), so it is stored as the byte v after checking that the map is exact."""
    import tempfile
    import PIL.Image
    from dust3r.utils.image import load_images
    from dust3r_b200.utils.synth import synth_photo
    lut = torch.arange(256, dtype=torch.uint8).to(torch.float32).div(255).sub_(0.5).div_(0.5)
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        for k, (H, W, seed, size, square_ok) in enumerate(IMAGE_CASES):
            photo = synth_photo(H, W, seed)
            path = os.path.join(tmp, f'{k}.png')
            PIL.Image.fromarray(photo).save(path)
            view = load_images([path], size=size, square_ok=square_ok, verbose=False)[0]
            img = view['img'][0]                                     # (3, H2, W2) float32
            v = torch.round((img * 0.5 + 0.5) * 255).to(torch.uint8)
            assert torch.equal(lut[v.long()], img), 'reference output is not one of the 256 normalised byte values'
            res[f'{k}|in'] = photo
            res[f'{k}|out_u8'] = v.permute(1, 2, 0).contiguous().numpy()
            res[f'{k}|true_shape'] = view['true_shape']
            res[f'{k}|args'] = np.int64([size, int(square_ok)])
            print('image', k, (H, W), '->', tuple(img.shape), 'size', size)
    np.savez_compressed(os.path.join(HERE, 'load_images.npz'), **res)


if __name__ == '__main__':
    what = sys.argv[1:] or ['pairs', 'align', 'forward', 'images']
    if 'images' in what:
        image_goldens()
    with torch.no_grad():
        if 'pairs' in what:
            pair_goldens()
    if 'align' in what:
        align_goldens()
    with torch.no_grad():
        if 'forward' in what:
            forward_goldens()
        if 'forward' in what or 'mixed' in what:
            forward_mixed_goldens()
        if 'forward' in what or 'odd' in what:
            forward_odd_grid_goldens()
