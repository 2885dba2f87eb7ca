"""load_images preprocessing (SURVEY §8f rank 4; dust3r/utils/image.py:62-128), CPU side:

  * oracle/image_oracle.py (integer restatement of Pillow's resize + crop + torchvision ImgNorm) is pinned bit-exactly against
    Pillow / torchvision themselves, the unmodified reference's load_images (its outputs recorded as digests in
    tests/golden/reference_records.npz) and the committed golden fixture tests/golden/load_images.npz (reference outputs);
  * the product's host-side tables (dust3r_b200/utils/image.py) equal the oracle's;
  * the per-thread bodies of the CUDA kernels (dust3r_b200/csrc/resample_core.h) are compiled for the HOST
    (tests/native/resample_host.cpp, g++) and run over every thread index of the launches: bit-exact against the host PIL
    pipeline, so the code the GPU executes is verified without a GPU.  The `-m gpu` twin is tests/test_scene_preprocess_gpu.py.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, digest, reference_records
from dust3r_b200.utils import image as img_mod
from dust3r_b200.utils.synth import synth_photo
from oracle import image_oracle as io

CASES = [  # (H, W, size, square_ok)
    (150, 200, 128, False), (200, 150, 128, False), (130, 130, 128, False), (130, 130, 128, True), (37, 53, 224, False),
    (300, 170, 224, False), (480, 640, 512, False), (640, 480, 512, False), (90, 70, 160, False), (384, 512, 512, False),
    (97, 1003, 512, False), (601, 397, 224, False), (224, 224, 224, False),
]


def _write_png(tmp_path, arr, name):
    import PIL.Image
    path = os.path.join(str(tmp_path), name)
    PIL.Image.fromarray(arr).save(path)
    return path


@pytest.mark.parametrize('method', [io.LANCZOS, io.BICUBIC])
def test_resize_oracle_equals_pillow(method):
    import PIL.Image
    pil_method = {io.LANCZOS: PIL.Image.LANCZOS, io.BICUBIC: PIL.Image.BICUBIC}[method]
    rng = np.random.default_rng(0)
    for k, (h, w, nh, nw) in enumerate([(37, 53, 24, 31), (200, 300, 64, 48), (48, 64, 100, 130), (480, 640, 384, 512),
                                        (100, 100, 100, 57), (57, 100, 57, 33), (31, 17, 224, 409), (1200, 900, 512, 384)]):
        for img in (rng.integers(0, 256, (h, w, 3), dtype=np.uint8), synth_photo(h, w, seed=k)):
            got = io.resize_u8(img, nw, nh, method)
            ref = np.asarray(PIL.Image.fromarray(img).resize((nw, nh), pil_method))
            assert np.array_equal(got, ref), (h, w, nh, nw, method)


def test_normalisation_equals_torchvision_for_every_byte():
    import torchvision.transforms as tvf
    import PIL.Image
    norm = tvf.Compose([tvf.ToTensor(), tvf.Normalize((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))])
    ramp = np.arange(256, dtype=np.uint8).reshape(16, 16, 1).repeat(3, axis=2)
    ref = norm(PIL.Image.fromarray(ramp))
    assert np.array_equal(io.normalise(ramp), ref.numpy())
    lut = img_mod.norm_lut()
    assert torch.equal(lut[torch.from_numpy(ramp).long()].permute(2, 0, 1), ref)
    assert float(lut[0]) == -1.0 and float(lut[255]) == 1.0


def test_product_tables_equal_oracle_tables():
    for a, b in [(53, 31), (300, 48), (64, 130), (640, 512), (480, 384), (100, 57), (4000, 512), (3000, 384), (17, 409),
                 (1024, 224), (683, 299), (2, 512), (5000, 1)]:
        for method in (io.LANCZOS, io.BICUBIC):
            b1, k1 = img_mod.resample_table(a, b, method)
            b2, k2 = io.coefficients(a, b, method)
            assert np.array_equal(b1, b2) and np.array_equal(k1, k2), (a, b, method)
            assert b1.dtype == np.int32 and k1.dtype == np.int32
    for (h, w, size, sq) in CASES:
        assert img_mod.resized_shape(w, h, size) == io.resized_shape(w, h, size)
        nw, nh, _ = io.resized_shape(w, h, size)
        assert img_mod._crop_box_int(nw, nh, size, sq) == io.crop_box(nw, nh, size, sq)
    # an unchanged dimension: identity table, which reproduces every byte
    bounds, coefs = img_mod.resample_table(77, 77, io.LANCZOS)
    assert np.array_equal(bounds[:, 0], np.arange(77)) and (bounds[:, 1] == 1).all() and (coefs == 1 << 22).all()


def test_oracle_equals_golden_reference_outputs():
    gold = np.load(os.path.join(GOLDEN, 'load_images.npz'))
    n = len([k for k in gold.files if k.endswith('|in')])
    assert n >= 8
    lut = img_mod.norm_lut().numpy()
    for k in range(n):
        size, square_ok = (int(v) for v in gold[f'{k}|args'])
        out, true_shape = io.load_image_oracle(gold[f'{k}|in'], size, bool(square_ok))
        ref = np.moveaxis(lut[gold[f'{k}|out_u8']], -1, 0)[None]
        assert np.array_equal(true_shape, gold[f'{k}|true_shape'])
        assert out.shape == ref.shape and np.array_equal(out, ref), k


def test_oracle_and_host_port_equal_live_reference_load_images(tmp_path):
    """The reference's load_images on the same PNG files, recorded in tests/golden/reference_records.npz (the image as a
    digest: ours must equal it bit for bit, and the oracle must equal ours)."""
    gold = reference_records()
    for k, (h, w, size, sq) in enumerate(CASES):
        ref = lambda key: gold[f'load_images|{k}|{key}']
        photo = synth_photo(h, w, seed=10 + k)
        assert digest(photo) == str(ref('photo')), ('synthetic photo differs from the recorded one', h, w)
        path = _write_png(tmp_path, photo, f'{k}.png')
        ours = img_mod.load_images([path], size=size, square_ok=sq, verbose=False)[0]
        out, true_shape = io.load_image_oracle(photo, size, sq)
        assert digest(ours['img']) == str(ref('img')) and np.array_equal(ours['true_shape'], ref('true_shape'))
        assert np.array_equal(out, ours['img'].numpy()) and np.array_equal(true_shape, ref('true_shape')), (h, w, size, sq)
        assert ours['idx'] == int(ref('idx')) and ours['instance'] == str(ref('instance'))


# ------------------------------------------------------------------------------------------------ the GPU code, on the host
@pytest.fixture(scope='module')
def host_kernels(tmp_path_factory):
    gxx = shutil.which('g++')
    if gxx is None:
        pytest.skip('no g++')
    out = os.path.join(str(tmp_path_factory.mktemp('native')), 'resample_host.so')
    src = os.path.join(ROOT, 'tests', 'native', 'resample_host.cpp')
    subprocess.run([gxx, '-O2', '-std=c++17', '-shared', '-fPIC', '-Wall', '-Wextra', '-Werror', '-o', out, src], check=True)
    lib = ctypes.CDLL(out)
    vp, i32 = ctypes.c_void_p, ctypes.c_int32
    lib.resample_host.restype = ctypes.c_int
    lib.resample_host.argtypes = [vp, i32, i32, i32, i32, vp, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp]
    return lib


def _run_on_host(lib, photo, size, square_ok):
    """What preprocess_image_u8 does, with host buffers and the host-compiled kernel bodies."""
    h0, w0 = photo.shape[:2]
    plan = img_mod.preprocess_plan(h0, w0, size, square_ok)
    xb, xk = img_mod.resample_table(w0, plan['w1'], plan['method'])
    yb, yk = img_mod.resample_table(h0, plan['h1'], plan['method'])
    lut = img_mod.norm_lut().numpy()
    src = np.ascontiguousarray(photo)
    tmp = np.full((plan['rows'], plan['w2'], 3), 0xAB, dtype=np.uint8)
    out = np.full((1, 3, plan['h2'], plan['w2']), np.nan, dtype=np.float32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    xk_t, yk_t = np.ascontiguousarray(xk.T), np.ascontiguousarray(yk.T)          # tap-major, as uploaded by _device_table
    rc = lib.resample_host(p(src), h0, w0, plan['h1'], plan['w1'], p(xb), p(xk_t), xk.shape[1], p(yb), p(yk_t), yk.shape[1],
                           plan['row0'], plan['rows'], plan['left'], plan['upper'], plan['h2'], plan['w2'], p(lut), p(tmp), p(out))
    assert rc == 0
    return out, plan


def test_kernel_bodies_on_host_equal_pillow_pipeline(host_kernels, tmp_path):
    """resample_core.h (what csrc/image_ops.cu launches) vs the host PIL pipeline of load_images, bit for bit."""
    for k, (h, w, size, sq) in enumerate(CASES + [(1500, 2000, 512, False), (2000, 1500, 224, False)]):
        photo = synth_photo(h, w, seed=20 + k)
        got, plan = _run_on_host(host_kernels, photo, size, sq)
        path = _write_png(tmp_path, photo, f'{k}.png')
        ref = img_mod.load_images([path], size=size, square_ok=sq, verbose=False)[0]
        assert got.shape == tuple(ref['img'].shape), (h, w, size, sq, plan)
        assert np.array_equal(got, ref['img'].numpy()), (h, w, size, sq)
        assert 0 <= plan['row0'] and plan['row0'] + plan['rows'] <= h


def test_kernel_bodies_on_host_equal_golden(host_kernels):
    gold = np.load(os.path.join(GOLDEN, 'load_images.npz'))
    lut = img_mod.norm_lut().numpy()
    for k in range(len([f for f in gold.files if f.endswith('|in')])):
        size, square_ok = (int(v) for v in gold[f'{k}|args'])
        got, _ = _run_on_host(host_kernels, gold[f'{k}|in'], size, bool(square_ok))
        assert np.array_equal(got, np.moveaxis(lut[gold[f'{k}|out_u8']], -1, 0)[None]), k


def test_preprocess_rejects_bad_input():
    with pytest.raises(ValueError):
        img_mod.preprocess_plan(3, 400, 512)          # resized to 4 x 512: nothing is left after the crop to multiples of 16
    from dust3r_b200 import _lib
    with pytest.raises(_lib.D3RError):
        img_mod.preprocess_image_u8(np.zeros((32, 32, 3), dtype=np.uint8), 512, device='cpu')   # no CPU fallback


def test_load_images_folder_threads_keep_the_sequential_contract(tmp_path, capsys):
    """Decoding on a thread pool must not change anything observable: file order, idx / instance, skipped files, verbose lines."""
    import PIL.Image
    shapes = [(90, 120), (120, 90), (100, 100), (64, 200), (33, 47), (150, 151), (80, 81)]
    for k, (h, w) in enumerate(shapes):
        PIL.Image.fromarray(synth_photo(h, w, seed=50 + k)).save(os.path.join(str(tmp_path), f'im{k:02d}.{"png" if k % 2 else "jpg"}'))
    open(os.path.join(str(tmp_path), 'readme.txt'), 'w').write('not an image')
    seq = img_mod.load_images(str(tmp_path), size=64, verbose=True, workers=1)
    lines_seq = capsys.readouterr().out
    for workers in (2, 3, None):
        par = img_mod.load_images(str(tmp_path), size=64, verbose=True, workers=workers)
        assert capsys.readouterr().out == lines_seq
        assert len(par) == len(seq) == len(shapes)
        for a, b in zip(par, seq):
            assert torch.equal(a['img'], b['img']) and np.array_equal(a['true_shape'], b['true_shape'])
            assert a['idx'] == b['idx'] and a['instance'] == b['instance']
    assert [v['idx'] for v in seq] == list(range(len(shapes))) and lines_seq.count(' - adding im') == len(shapes)
    # the reference's load_images on the same folder (recorded in tests/golden/reference_records.npz)
    gold = reference_records()
    assert [digest(a['img']) for a in seq] == gold['load_images_folder|img'].tolist()
    assert np.array_equal(np.concatenate([a['true_shape'] for a in seq]), gold['load_images_folder|true_shape'])
    assert [a['instance'] for a in seq] == gold['load_images_folder|instance'].tolist()
    with pytest.raises(AssertionError):
        img_mod.load_images([os.path.join(str(tmp_path), 'readme.txt')], size=64, verbose=False)
