"""The oracles against the committed golden vectors made by the reference itself.  CPU only."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, digest, reference_records
from dust3r_b200.utils.synth import synth_state_dict, synth_images, synth_pair_predictions
from dust3r_b200.image_pairs import make_pairs
from oracle.forward_oracle import forward_oracle
from oracle.align_oracle import AlignProblem, init_params, align_oracle


def _small_cfgs():
    import importlib.util
    spec = importlib.util.spec_from_file_location('make_golden_cfg', os.path.join(GOLDEN, 'make_golden.py'))
    src = open(os.path.join(GOLDEN, 'make_golden.py')).read()
    # only the SMALL table is needed; evaluate it without importing the reference
    from dust3r_b200.config import ModelConfig
    ns = {'ModelConfig': ModelConfig}
    start = src.index('SMALL = dict(')
    end = src.index('\n)\n', start) + 3
    exec(src[start:end], ns)
    return ns['SMALL']


def _forward_case(name):
    """(cfg, H, W) of a forward golden: a SMALL entry, or 'small_dpt_{H}x{W}' for the odd token grids of make_golden.py"""
    if name in _small_cfgs():
        return _small_cfgs()[name]
    base, size = name.rsplit('_', 1)
    H, W = (int(v) for v in size.split('x'))
    return _small_cfgs()[base][0], H, W


def _run_oracle_like_inference(cfg, sd, pairs, batch_size):
    """inference() semantics (inference.py:55-72): batches of `batch_size` pairs, outputs concatenated."""
    res = {k: [] for k in ('pts3d', 'conf1', 'pts3d_in_other_view', 'conf2')}
    for i in range(0, len(pairs), batch_size):
        chunk = pairs[i:i + batch_size]
        img1 = torch.cat([a['img'] for a, b in chunk])
        img2 = torch.cat([b['img'] for a, b in chunk])
        r1, r2 = forward_oracle(sd, cfg, img1, img2, [a['instance'] for a, b in chunk], [b['instance'] for a, b in chunk])
        res['pts3d'].append(r1['pts3d']); res['conf1'].append(r1['conf'])
        res['pts3d_in_other_view'].append(r2['pts3d_in_other_view']); res['conf2'].append(r2['conf'])
    return {k: torch.cat(v) for k, v in res.items()}


@pytest.mark.parametrize('name', ['small_dpt', 'small_linear', 'small_dpt_48x80', 'small_dpt_80x48'])
def test_forward_oracle_matches_reference_golden(name):
    """small_dpt_48x80 / _80x48: token grids of odd width / height (3 x 5, 5 x 3) through the DPT head"""
    cfg, H, W = _forward_case(name)
    gold = np.load(os.path.join(GOLDEN, f'forward_{name}.npz'))
    sd = synth_state_dict(cfg, seed=11)
    imgs = synth_images(3, H, W, seed=5)
    assert np.allclose([float(i['img'].double().sum()) for i in imgs], gold['img_sum'], rtol=1e-9), \
        'synthetic inputs differ from the ones the golden was made with'
    pairs = make_pairs(imgs, scene_graph='complete', prefilter=None, symmetrize=True)
    assert [a['idx'] for a, b in pairs] == gold['idx1'].tolist() and [b['idx'] for a, b in pairs] == gold['idx2'].tolist()
    out = _run_oracle_like_inference(cfg, sd, pairs, 4)
    for k in ('pts3d', 'conf1', 'pts3d_in_other_view', 'conf2'):
        ref = torch.from_numpy(gold[k])
        assert out[k].shape == ref.shape
        # identical torch ops on the same machine family: allow only accumulation-order noise
        assert torch.allclose(out[k], ref, rtol=2e-4, atol=2e-5), (k, float((out[k] - ref).abs().max()))


def _mixed_size_pairs(H, W):
    sizes = [(H, W), (H - 16, W), (H, W - 32)]
    imgs = [dict(synth_images(1, h, w, seed=20 + k)[0], idx=k, instance=str(k)) for k, (h, w) in enumerate(sizes)]
    return make_pairs(imgs, scene_graph='complete', prefilter=None, symmetrize=True)


@pytest.mark.parametrize('name', ['small_dpt', 'small_linear'])
def test_forward_oracle_mixed_sizes_matches_reference_golden(name):
    """Pairs whose two images differ in size: the reference runs them one pair per call and encodes the two views
    separately (inference.py:60-64, model.py:147-151); fixtures made by the unmodified reference."""
    cfg, H, W = _small_cfgs()[name]
    sd = synth_state_dict(cfg, seed=11)
    pairs = _mixed_size_pairs(H, W)
    gold = np.load(os.path.join(GOLDEN, f'forward_{name}_mixed.npz'))
    assert [a['idx'] for a, b in pairs] == gold['idx1'].tolist() and [b['idx'] for a, b in pairs] == gold['idx2'].tolist()
    for k, (a, b) in enumerate(pairs):
        r1, r2 = forward_oracle(sd, cfg, a['img'], b['img'], [a['instance']], [b['instance']])
        for got, key in ((r1['pts3d'][0], f'pts3d_{k}'), (r1['conf'][0], f'conf1_{k}'),
                         (r2['pts3d_in_other_view'][0], f'pts3d_in_other_view_{k}'), (r2['conf'][0], f'conf2_{k}')):
            ref = torch.from_numpy(gold[key])
            assert got.shape == ref.shape
            assert (got - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item()), (key, (got - ref).abs().max().item())


def test_forward_oracle_matches_reference_golden_vitl_224_linear():
    from dust3r_b200.config import vitl_224_linear
    cfg = vitl_224_linear()
    gold = np.load(os.path.join(GOLDEN, 'forward_vitl_224_linear.npz'))
    sd = synth_state_dict(cfg, seed=0)
    imgs = synth_images(2, 224, 224, seed=3)
    r1, r2 = forward_oracle(sd, cfg, imgs[0]['img'], imgs[1]['img'], ['0'], ['1'])
    s = int(gold['stride'])
    for got, k in ((r1['pts3d'], 'pts3d'), (r1['conf'], 'conf1'), (r2['pts3d_in_other_view'], 'pts3d_in_other_view'), (r2['conf'], 'conf2')):
        ref = torch.from_numpy(gold[k])
        assert torch.allclose(got[:, ::s, ::s], ref, rtol=1e-3, atol=1e-4), (k, float((got[:, ::s, ::s] - ref).abs().max()))


def _edges(n):
    e = [(i, j) for i in range(n) for j in range(i)]
    return e + [(j, i) for i, j in e]


@pytest.mark.parametrize('variant', ['stacked', 'per_edge'])
@pytest.mark.parametrize('dist', ['l1', 'l2'])
@pytest.mark.parametrize('schedule', ['cosine', 'linear'])
def test_align_oracle_matches_reference_golden(variant, dist, schedule):
    """golden = unmodified reference loop + local roma restatement (see oracle/roma_stub)."""
    gold = np.load(os.path.join(GOLDEN, 'align_n4.npz'))
    n, H, W = 4, 24, 32
    out = synth_pair_predictions(n, _edges(n), H, W, seed=1)
    prob = AlignProblem.from_output(out, dist=dist, variant=variant)
    P0 = init_params(prob, seed=5)
    losses, final = align_oracle(prob, P0, niter=60, schedule=schedule)
    key = f'{variant}|{dist}|{schedule}'
    ref = gold[key + '|loss']
    assert np.allclose(losses, ref, rtol=2e-5), float(np.abs(np.array(losses) / ref - 1).max())
    assert np.allclose(torch.stack(final['im_depthmaps']).numpy(), gold[key + '|depth'], atol=2e-4)
    assert np.allclose(final['im_poses'].numpy(), gold[key + '|poses'], atol=2e-4)
    assert np.allclose(final['pw_poses'].numpy(), gold[key + '|pw'], atol=2e-4)
    assert np.allclose(final['im_focals'].numpy(), gold[key + '|focals'], atol=2e-4)


def test_forward_oracle_bit_matches_live_reference():
    """A symmetrised batch (the reference's half-encoder path) against the reference model's outputs, recorded at a fixed
    quarter of the pixels in tests/golden/reference_records.npz."""
    from dust3r_b200.config import ModelConfig
    gold = reference_records()
    cfg = ModelConfig(img_size=(64, 64), enc_embed_dim=128, enc_depth=2, enc_num_heads=2, dec_embed_dim=64,
                      dec_depth=10, dec_num_heads=1, head_type='dpt', landscape_only=False)
    sd = synth_state_dict(cfg, seed=21)
    imgs = synth_images(4, 48, 64, seed=9)
    img1 = torch.cat([imgs[0]['img'], imgs[1]['img']])
    img2 = torch.cat([imgs[1]['img'], imgs[0]['img']])
    assert digest(img1) + digest(img2) == str(gold['forward_sym|inputs']), 'synthetic inputs differ from the recorded ones'
    o1, o2 = forward_oracle(sd, cfg, img1, img2, ['0', '1'], ['1', '0'])
    px = torch.from_numpy(gold['forward_sym|px'])
    for got, key in ((o1['pts3d'], 'pts3d'), (o1['conf'], 'conf1'), (o2['pts3d_in_other_view'], 'pts3d_in_other_view'),
                     (o2['conf'], 'conf2')):
        ref = torch.from_numpy(gold[f'forward_sym|{key}'])
        assert torch.allclose(ref, got.reshape(2, 48 * 64, -1)[:, px], rtol=1e-5, atol=1e-6), key


@pytest.mark.parametrize('name', ['small_linear', 'small_dpt'])
def test_many_ar_golden_equals_oracle_on_untransposed_items(name):
    """landscape_only=True (ManyAR_PatchEmbed + transpose_to_landscape.wrapper_yes, utils/misc.py:66-95): for a portrait item
    stored transposed in a landscape batch the reference returns transpose(model(un-transposed image)).  Checked item by item
    against the oracle on the golden produced by the unmodified reference (tests/golden/make_golden.py::many_ar_golden)."""
    gold = np.load(os.path.join(GOLDEN, f'forward_{name}_manyar.npz'))
    H, W = int(gold['H']), int(gold['W'])
    from dust3r_b200.utils.synth import many_ar_inputs
    v1, v2 = many_ar_inputs(H, W)
    cfg = _small_cfgs()[name][0]
    sd = synth_state_dict(cfg, seed=11)
    for k in range(4):
        p1, p2 = bool(v1['true_shape'][k, 0] > v1['true_shape'][k, 1]), bool(v2['true_shape'][k, 0] > v2['true_shape'][k, 1])
        a, b = v1['img'][k:k + 1], v2['img'][k:k + 1]
        o1, o2 = forward_oracle(sd, cfg, a.swapaxes(-1, -2) if p1 else a, b.swapaxes(-1, -2) if p2 else b)
        for got, port, key in ((o1['pts3d'], p1, 'pts3d'), (o1['conf'], p1, 'conf1'),
                               (o2['pts3d_in_other_view'], p2, 'pts3d_in_other_view'), (o2['conf'], p2, 'conf2')):
            got = got.swapaxes(1, 2) if port else got
            ref = torch.from_numpy(gold[key][k:k + 1])
            assert got.shape == ref.shape
            assert float((got - ref).abs().max()) <= 2e-5 * float(ref.abs().max()), (name, k, key)
