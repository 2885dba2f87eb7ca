"""The forward path's kernels one at a time, through the C ABI, against float64 references computed from the same bf16- or
fp32-rounded inputs the kernel reads.

Bounds (DESIGN.md section 2):
  * data movement (patch im2col, gather, stride-2 im2col, fp32 -> bf16 cast) and the linear head's linear mode: bit-exact;
  * GEMM-like kernels, every element: |y - y_ref| <= 2^-8 |y_ref| + GAMMA (|A| |B|^T), |A| |B|^T being the same contraction
    over absolute values (one bf16 rounding of the output, plus fp32 accumulation);
  * bilinear x2 upsampling and LayerNorm: 1 bf16 ulp of the reference, plus, for results near zero, the fp32 rounding the
    kernel cannot avoid: of the source coordinates (2^-20 max(H, W) max|x|) / of the row mean, which 1 / std amplifies
    (2^-17 |mean| rstd |g|), and of the affine transform (2^-16 (|x_hat g| + |b|));
  * fp32 postprocess formulas: a few fp32 ulps, stated per formula below.
The tests with a bound print their worst error / bound ratio."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from dust3r_b200 import _lib
from dust3r_b200.model import pack_conv3x3, pack_conv3x3_s2, pack_convT

pytestmark = pytest.mark.gpu

# fp32 accumulation term of the GEMM bound.  Measured on a B200 (1000 W power limit): no element needs more than 3.9e-7
# beyond the bf16 rounding term (stride-2 conv at 21 x 32, K = 6912; _gamma_needed), 600x below GAMMA; worst ratio to the
# whole bound 0.91 (transposed conv k = 4), which the bf16 rounding of the output dominates.
GAMMA = 2.0 ** -12
# the head tail never rounds through bf16 (fp32 accumulator, fp32 w4, fp32 output): its bound is GAMMA_HEAD |w4| (conv(|x|, |W|)
# + |bias|) + |b4| plus a few fp32 ulps.  Measured on a B200: no element needs more than 7e-7 of that magnitude, 5x below
# GAMMA_HEAD; rounding relu(conv) to bf16 before the 1x1 conv would need about 2^-12.
GAMMA_HEAD = 2.0 ** -18
ULP32 = 2.0 ** -24


@pytest.fixture(params=[0, 1], ids=['cta1', 'cta_pair'])
def gemm_impl(request):
    """the GEMM-like tests run on both kernel families: 1-CTA tcgen05 and CTA-pair (cta_group::2)"""
    lib = _lib.get_lib()
    lib.d3r_set_gemm_impl(request.param)
    yield request.param
    lib.d3r_set_gemm_impl(2)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _rand(shape, dev, scale=1.0, seed=0):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


def _sync_check(rc):
    _lib.check(rc)
    torch.cuda.synchronize()


def _ratio(err, bound):
    """worst err / bound over all elements (bound > 0 everywhere)"""
    return float((err / bound).max())


def _gamma_needed(out, ref, mag):
    """smallest GAMMA the elements need beyond the bf16 rounding term (<= 0: rounding covers every element)"""
    return float((((out.double() - ref).abs() - 2 ** -8 * ref.abs()) / mag).max())


def _ulp_bf16(v):
    """spacing of bf16 numbers at |v| (8 significant bits), v float64; at v = 0 the smallest bf16 subnormal"""
    _, e = torch.frexp(v.abs())
    return torch.where(v == 0, torch.full_like(v, 2.0 ** -133), torch.ldexp(torch.ones_like(v), e - 8))


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


# ---- bit-exact data movement ------------------------------------------------------------------------------------------

@pytest.mark.parametrize('B,H,W', [(1, 16, 16), (2, 48, 80), (3, 80, 48), (1, 32, 336)])
def test_patch_im2col16_is_unfold(cuda_device, B, H, W):
    lib = _lib.get_lib()
    img = _rand((B, 3, H, W), cuda_device, seed=1)
    L = (H // 16) * (W // 16)
    out = torch.full((B * L, 768), float('nan'), dtype=torch.bfloat16, device=cuda_device)
    _sync_check(lib.d3r_patch_im2col16(_p(img), _p(out), B, H, W, _lib.stream_ptr()))
    ref = F.unfold(img, 16, stride=16).transpose(1, 2).reshape(B * L, 768).bfloat16()
    assert torch.equal(out, ref)


def test_gather_images_repeated_and_out_of_order(cuda_device):
    lib = _lib.get_lib()
    n_in, rows, Cc = 5, 15, 136
    src = _rand((n_in * rows, Cc), cuda_device, seed=2).bfloat16()
    for mp in ([4, 0, 4, 2, 2, 1, 3, 0], [3], [0, 1, 2, 3, 4]):
        m = torch.tensor(mp, dtype=torch.int32, device=cuda_device)
        out = torch.full((len(mp) * rows, Cc), float('nan'), dtype=torch.bfloat16, device=cuda_device)
        _sync_check(lib.d3r_gather_images_bf16(_p(src), _p(out), _p(m), len(mp), rows, Cc, _lib.stream_ptr()))
        ref = src.view(n_in, rows, Cc)[m.long()].reshape(-1, Cc)
        assert torch.equal(out, ref), mp


def _im2col_s2(x):
    lib = _lib.get_lib()
    B, H, W, Cc = x.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.full((B * Ho * Wo, 9 * Cc), float('nan'), dtype=torch.bfloat16, device=x.device)
    _sync_check(lib.d3r_im2col_3x3_s2_bf16(_p(x), _p(out), B, H, W, Cc, _lib.stream_ptr()))
    return out, Ho, Wo


@pytest.mark.parametrize('B,H,W,Cc', [(2, 3, 5, 768), (2, 5, 3, 768), (1, 4, 6, 768), (2, 21, 32, 64), (2, 32, 21, 64),
                                      (1, 1, 1, 8), (3, 2, 7, 16)])
def test_im2col_3x3_s2_is_unfold(cuda_device, B, H, W, Cc):
    x = _rand((B, H, W, Cc), cuda_device, seed=3).bfloat16()
    out, Ho, Wo = _im2col_s2(x)
    # unfold columns are (c, tap): reorder to the kernel's (tap, c)
    ref = F.unfold(_nchw(x.float()), 3, padding=1, stride=2).view(B, Cc, 9, Ho * Wo).permute(0, 3, 2, 1)
    assert torch.equal(out, ref.reshape(B * Ho * Wo, 9 * Cc).bfloat16())


def test_cast_f32_bf16_rounds_to_nearest_even(cuda_device):
    lib = _lib.get_lib()
    bits = []
    for m in (0x3F80, 0x3F81, 0xBF80, 0xBF81, 0x0001, 0x7F00, 0x7F7F):   # ties to even (down and up), both signs, subnormal
        bits += [(m << 16) | 0x8000, (m << 16) | 0x7FFF, (m << 16) | 0x8001]
    bits += [0x00000000, 0x80000000,                         # +-0
             0x00000001, 0x80000001, 0x007FFFFF, 0x00400000,  # fp32 subnormals
             0x00008000, 0x00018000,                          # subnormal exact ties
             0x7F800000, 0xFF800000,                          # +-inf
             0x7F7FFFFF, 0xFF7FFFFF, 0x7F7F8000, 0x7F7F7FFF,  # above the bf16 maximum (rounds to inf) and just below
             0x7FC00000, 0xFFC00001, 0x7F800001]              # NaNs
    rnd = torch.randint(-2 ** 31, 2 ** 31 - 1, (4096,), generator=torch.Generator().manual_seed(4), dtype=torch.int64)
    allbits = torch.tensor(bits, dtype=torch.int64)
    allbits = torch.cat((allbits, rnd))
    allbits = allbits[:allbits.numel() // 4 * 4]
    x = ((allbits + 2 ** 31) % 2 ** 32 - 2 ** 31).to(torch.int32).view(torch.float32)
    out = torch.full(x.shape, 7.0, dtype=torch.bfloat16, device=cuda_device)
    xd = x.to(cuda_device)
    _sync_check(lib.d3r_cast_f32_bf16(_p(xd), _p(out), x.numel(), _lib.stream_ptr()))
    # round to nearest even on the bit pattern (exact for subnormals, overflows to inf past the bf16 maximum)
    u = x.view(torch.int32).to(torch.int64) % 2 ** 32
    ref = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) % 2 ** 16).to(torch.int32)
    got = out.cpu().view(torch.int16).to(torch.int32) % 2 ** 16
    nan = torch.isnan(x)
    assert torch.isnan(out.cpu()[nan].float()).all()
    assert torch.equal(got[~nan], ref[~nan])


# ---- GEMM-like kernels --------------------------------------------------------------------------------------------------

CONVT_CASES = [(4, 96, 96, h, w) for h, w in ((3, 5), (5, 3), (21, 32), (32, 21))] + \
              [(2, 192, 192, h, w) for h, w in ((3, 5), (5, 3), (21, 32), (32, 21))]


@pytest.mark.timeout(300)
@pytest.mark.parametrize('k,Cin,Cout,h,w', CONVT_CASES)
def test_convT_matches_conv_transpose2d(cuda_device, gemm_impl, k, Cin, Cout, h, w):
    """act_postprocess 0 / 1 (k = stride = 4 / 2) with the product's weight packing; M = 2 h w is not a multiple of 128."""
    lib = _lib.get_lib()
    B = 2
    x = _rand((B, h, w, Cin), cuda_device, seed=5).bfloat16()
    wt = _rand((Cin, Cout, k, k), cuda_device, scale=Cin ** -0.5, seed=6).bfloat16()     # ConvTranspose2d layout
    bias = _rand((Cout,), cuda_device, seed=7)
    out = torch.full((B, h * k, w * k, Cout), float('nan'), dtype=torch.bfloat16, device=cuda_device)
    wp = pack_convT(wt)
    _sync_check(lib.d3r_convT_bf16(_p(x), _p(wp), _p(bias), _p(out), B, h, w, Cin, Cout, k, _lib.stream_ptr()))
    ref = _nhwc(F.conv_transpose2d(_nchw(x.double()), wt.double(), bias.double(), stride=k))
    mag = _nhwc(F.conv_transpose2d(_nchw(x.double().abs()), wt.double().abs(), stride=k))
    r = _ratio((out.double() - ref).abs(), 2 ** -8 * ref.abs() + GAMMA * mag)
    print(f'convT k={k} C={Cin} {h}x{w} impl={gemm_impl}: worst ratio {r:.3e}, gamma needed {_gamma_needed(out, ref, mag):.2e}')
    assert r <= 1.0, r


@pytest.mark.timeout(300)
@pytest.mark.parametrize('h,w', [(3, 5), (5, 3), (4, 6), (21, 32), (32, 21)])
def test_stride2_conv_matches_conv2d(cuda_device, gemm_impl, h, w):
    """act_postprocess 3: im2col (3x3, stride 2, pad 1) + GEMM with the packed [768][9*768] weight, on odd and even grids."""
    lib = _lib.get_lib()
    B, Cc = 2, 768
    x = _rand((B, h, w, Cc), cuda_device, seed=8).bfloat16()
    wt = _rand((Cc, Cc, 3, 3), cuda_device, scale=(9 * Cc) ** -0.5, seed=9).bfloat16()
    bias = _rand((Cc,), cuda_device, seed=10)
    col, Ho, Wo = _im2col_s2(x)
    wp = pack_conv3x3_s2(wt).contiguous()
    M, K = B * Ho * Wo, 9 * Cc
    out = torch.full((M, Cc), float('nan'), dtype=torch.bfloat16, device=cuda_device)
    _sync_check(lib.d3r_gemm_bf16(_p(col), _p(wp), _p(out), _p(bias), None, None, M, Cc, K, Cc, 1, None, None, 0, 0, 0,
                                  _lib.stream_ptr()))
    ref = _nhwc(F.conv2d(_nchw(x.double()), wt.double(), bias.double(), stride=2, padding=1)).reshape(M, Cc)
    mag = _nhwc(F.conv2d(_nchw(x.double().abs()), wt.double().abs(), stride=2, padding=1)).reshape(M, Cc)
    r = _ratio((out.double() - ref).abs(), 2 ** -8 * ref.abs() + GAMMA * mag)
    print(f'stride-2 conv {h}x{w} impl={gemm_impl}: worst ratio {r:.3e}, gamma needed {_gamma_needed(out, ref, mag):.2e}')
    assert r <= 1.0, r


def _depth_ref(xyz, mode):
    """heads/postprocess.py reg_dense_depth, float64"""
    if mode == 0:
        return xyz
    d = xyz.norm(dim=-1, keepdim=True)
    u = xyz / d.clamp_min(1e-8)
    return u * d.square() if mode == 1 else u * torch.expm1(d)


def _conf_ref(c, mode, cmin, cmax):
    """heads/postprocess.py reg_dense_conf, float64"""
    if mode == 1:
        return cmin + c.exp().clamp(max=cmax - cmin)
    return (cmax - cmin) * torch.sigmoid(c) + cmin


def _depth_bound(xyz, err, mode):
    """first-order propagation of a per-component bound `err` on xyz through reg_dense_depth: out_i = x_i g(d) with
    g = d (square) or expm1(d) / d (exp), |d out_i / d x_j| <= delta_ij g + |x_i| g'"""
    if mode == 0:
        return err
    d = xyz.norm(dim=-1, keepdim=True).clamp_min(1e-8)
    if mode == 1:
        g, gp = d, torch.ones_like(d)
    else:
        g = torch.expm1(d) / d
        gp = (torch.exp(d) * d - torch.expm1(d)) / d.square()
    return g * err + xyz.abs() * gp * err.sum(dim=-1, keepdim=True)


HEAD_MODES = [(0, 0), (0, 1), (0, 2), (1, 0), (1, 1), (1, 2), (2, 0), (2, 1), (2, 2)]
CONF_RANGE = {1: (1.0, 3.0e38), 2: (0.5, 4.0)}


@pytest.mark.timeout(600)
@pytest.mark.parametrize('H,W', [(48, 80), (80, 48), (32, 336)])
def test_conv3x3_head_tail_matches_float64(cuda_device, gemm_impl, H, W):
    """Last DPT conv + ReLU + 1x1 conv to 4 channels + postprocess, every depth mode (linear / square / exp) x conf mode
    (none / exp / sigmoid), with 4 channels (confidence) and with 3 (w4 row 3 zero, conf = NULL), on partial conv tiles.
    The linear xyz and the conf logit get GAMMA_HEAD times the magnitude |w4| (conv(|x|, |W|) + |bias|) + |b4| plus 8 fp32
    ulps (no bf16 term: nothing is rounded to bf16); square and exp carry it through the postprocess to first order and add
    the fp32 ulps of their own formulas (8 for square, 8 + 4 d for exp).  Conf logits here stay well below 88: beyond it exp(c) overflows and
    the reference returns an infinite conf, while the product clamps conf_max to 3.0e38 (model.py) and returns that."""
    lib = _lib.get_lib()
    B = 2
    x = _rand((B, H, W, 128), cuda_device, seed=11).bfloat16()
    wt = _rand((128, 128, 3, 3), cuda_device, scale=(9 * 128) ** -0.5, seed=12).bfloat16()
    bias = _rand((128,), cuda_device, scale=0.3, seed=13)
    w4 = _rand((4, 128), cuda_device, scale=0.2, seed=14)
    b4 = _rand((4,), cuda_device, seed=15)
    wp = pack_conv3x3(wt)
    conv = _nhwc(F.conv2d(_nchw(x.double()), wt.double(), bias.double(), padding=1))
    conv_mag = _nhwc(F.conv2d(_nchw(x.double().abs()), wt.double().abs(), padding=1)) + bias.double().abs()
    worst = 0.0
    for nch in (4, 3):
        w4n = w4.clone()
        b4n = b4.clone()
        if nch == 3:
            w4n[3] = 0
            b4n[3] = 0
        head = conv.relu() @ w4n.double().T + b4n.double()
        mag = conv_mag @ w4n.double().abs().T + b4n.double().abs()
        err = GAMMA_HEAD * mag + 8 * ULP32 * head.abs()
        xyz, c = head[..., :3], head[..., 3]
        assert float(c.max()) < 40
        for depth_mode, conf_mode in HEAD_MODES:
            for with_conf in ((True, False) if nch == 4 else (False,)):
                pts = torch.full((B, H, W, 3), float('nan'), device=cuda_device)
                conf = torch.full((B, H, W), float('nan'), device=cuda_device) if with_conf else None
                cmin, cmax = CONF_RANGE.get(conf_mode, (0.0, 0.0))
                _sync_check(lib.d3r_conv3x3_head_tail(_p(x), _p(wp), _p(bias), _p(w4n), _p(b4n), _p(pts), _p(conf), B, H, W,
                                                      depth_mode, conf_mode, cmin, cmax, _lib.stream_ptr()))
                ref = _depth_ref(xyz, depth_mode)
                d = xyz.norm(dim=-1, keepdim=True)
                own = 8 * ULP32 if depth_mode < 2 else (8 + 4 * d) * ULP32
                bound = _depth_bound(xyz, err[..., :3], depth_mode) + own * ref.abs() + 1e-45
                r = _ratio((pts.double() - ref).abs(), bound)
                assert r <= 1.0, (nch, depth_mode, conf_mode, with_conf, r)
                worst = max(worst, r)
                if with_conf and conf_mode:
                    cref = _conf_ref(c, conf_mode, cmin, cmax)
                    slope = c.exp() if conf_mode == 1 else (cmax - cmin) * torch.sigmoid(c) * torch.sigmoid(-c)
                    cb = slope * err[..., 3] + 8 * ULP32 * (cref.abs() + abs(cmin))
                    rc = _ratio((conf.double() - cref).abs(), cb)
                    assert rc <= 1.0, (nch, depth_mode, conf_mode, rc)
                    worst = max(worst, rc)
                elif with_conf:
                    assert torch.isnan(conf).all(), 'conf written with conf_mode 0'
    print(f'head tail {H}x{W} impl={gemm_impl}: worst ratio {worst:.3e}')


# ---- bandwidth-bound kernels with an ulp bound --------------------------------------------------------------------------

UPSAMPLE_CASES = [  # B, H, W, C, Ho, Wo
    (2, 1, 5, 8, 2, 10), (1, 3, 1, 8, 6, 2), (1, 1, 1, 128, 2, 2), (2, 2, 3, 256, 3, 5), (2, 3, 2, 256, 5, 3),
    (2, 11, 16, 256, 21, 32), (2, 16, 11, 256, 32, 21), (1, 7, 9, 128, 14, 18), (1, 13, 21, 128, 25, 41),
    (2, 24, 40, 128, 48, 80), (1, 5, 5, 8, 9, 10)]


@pytest.mark.parametrize('B,H,W,Cc,Ho,Wo', UPSAMPLE_CASES)
def test_upsample2x_matches_interpolate(cuda_device, B, H, W, Cc, Ho, Wo):
    """align_corners=True on the (2H, 2W) grid, cropped to Ho x Wo (refinenet4's crop); H or W = 1, odd sizes, Ho = 2H - 1
    and Ho not a multiple of the 8 rows a thread walks."""
    lib = _lib.get_lib()
    x = _rand((B, H, W, Cc), cuda_device, seed=16).bfloat16()
    out = torch.full((B, Ho, Wo, Cc), float('nan'), dtype=torch.bfloat16, device=cuda_device)
    _sync_check(lib.d3r_upsample2x_bf16(_p(x), _p(out), B, H, W, Cc, Ho, Wo, _lib.stream_ptr()))

    def up(t):
        return _nhwc(F.interpolate(_nchw(t), size=(2 * H, 2 * W), mode='bilinear', align_corners=True))[:, :Ho, :Wo]
    ref = up(x.double())
    bound = _ulp_bf16(ref) + 2 ** -20 * max(H, W) * float(x.abs().max())
    r = _ratio((out.double() - ref).abs(), bound)
    print(f'upsample {H}x{W}x{Cc} -> {Ho}x{Wo}: worst ratio {r:.3e}')
    assert r <= 1.0, r


def _ln_rows(kind, M, Cc, g):
    if kind == 'normal':
        return torch.randn((M, Cc), generator=g)
    if kind == 'offset':
        return 100 + torch.randn((M, Cc), generator=g)
    if kind == 'massive':
        x = torch.randn((M, Cc), generator=g)
        x[:, 3], x[:, Cc // 2 + 1] = 300.0, -300.0
        return x
    if kind == 'tiny_std':      # variance 1e-6: eps = 1e-6 matters
        return 0.5 + 1e-3 * torch.randn((M, Cc), generator=g)
    # constant rows (dyadic values: the fp32 row sum is exact, so x - mean is exactly 0)
    return torch.tensor([3.5, -1.25, 0.0, 1024.0])[torch.arange(M) % 4].view(M, 1).expand(M, Cc).contiguous()


@pytest.mark.parametrize('Cc', [64, 128, 768, 1024, 1280, 2048])
def test_layernorm_matches_float64(cuda_device, Cc):
    """Both register templates (C <= 1024 and above), M in {1, 7, 9, 1000}; N(0, 1) rows, an offset of 100, two massive
    activation channels at +-300, standard deviation 1e-3 (eps matters), constant rows (output exactly the bias)."""
    lib = _lib.get_lib()
    g = torch.Generator().manual_seed(Cc)
    gam = (1 + 0.5 * torch.randn((Cc,), generator=g)).to(cuda_device)
    bet = (0.5 * torch.randn((Cc,), generator=g)).to(cuda_device)
    worst = 0.0
    for M in (1, 7, 9, 1000):
        for kind in ('normal', 'offset', 'massive', 'tiny_std', 'constant'):
            x = _ln_rows(kind, M, Cc, g).to(cuda_device)
            out = torch.full((M, Cc), float('nan'), dtype=torch.bfloat16, device=cuda_device)
            _sync_check(lib.d3r_layernorm_bf16(_p(x), _p(gam), _p(bet), _p(out), M, Cc, 1e-6, _lib.stream_ptr()))
            xd = x.double()
            nrm = F.layer_norm(xd, (Cc,), eps=1e-6)
            ref = nrm * gam.double() + bet.double()
            rstd = (xd.var(dim=1, unbiased=False, keepdim=True) + 1e-6).rsqrt()
            bound = _ulp_bf16(ref) + 2 ** -16 * ((nrm * gam.double()).abs() + bet.double().abs()) + \
                2 ** -17 * xd.mean(dim=1, keepdim=True).abs() * rstd * gam.double().abs()
            r = _ratio((out.double() - ref).abs(), bound)
            assert r <= 1.0, (M, kind, r)
            worst = max(worst, r)
            if kind == 'constant':
                assert torch.equal(out, bet.bfloat16().expand(M, Cc)), M
    print(f'layernorm C={Cc}: worst ratio {worst:.3e}')


@pytest.mark.parametrize('nch', [3, 4])
def test_linear_head_postprocess_matches_float64(cuda_device, nch):
    """Pixel shuffle + heads/postprocess.py for every mode; zero and very short (|xyz| < 1e-8) vectors included.  The linear
    mode copies bit for bit.  fp32 bounds: square 8 ulp of |pts|; exp (8 + 4 d) ulp of |pts| (expm1 amplifies the error of
    d); confidence 8 ulp of |conf| + |conf_min|."""
    lib = _lib.get_lib()
    B, gh, gw = 2, 3, 5
    g = torch.Generator().manual_seed(17)
    feat = torch.randn((B * gh * gw, nch * 256), generator=g)
    f = feat.view(B * gh * gw, nch, 256)
    f[0, :3, :7] = 0                                         # zero vectors
    f[1, :3, :7] = 1e-9 * torch.randn((3, 7), generator=g)   # |xyz| < 1e-8
    feat = feat.to(cuda_device)
    H, W = gh * 16, gw * 16
    shuf = feat.double().view(B, gh, gw, nch, 16, 16).permute(0, 1, 4, 2, 5, 3).reshape(B, H, W, nch)
    xyz = shuf[..., :3]
    assert int((xyz.norm(dim=-1) < 1e-8).sum()) >= 14
    worst = 0.0
    for depth_mode, conf_mode in HEAD_MODES:
        pts = torch.full((B, H, W, 3), float('nan'), device=cuda_device)
        conf = torch.full((B, H, W), float('nan'), device=cuda_device) if nch == 4 else None
        cmin, cmax = CONF_RANGE.get(conf_mode, (0.0, 0.0))
        _sync_check(lib.d3r_linear_head_postprocess(_p(feat), _p(pts), _p(conf), B, gh, gw, nch, depth_mode, conf_mode,
                                                    cmin, cmax, _lib.stream_ptr()))
        ref = _depth_ref(xyz, depth_mode)
        if depth_mode == 0:
            assert torch.equal(pts.double(), ref)
        else:
            d = xyz.norm(dim=-1, keepdim=True)
            rel = 8 * ULP32 if depth_mode == 1 else (8 + 4 * d) * ULP32
            r = _ratio((pts.double() - ref).abs(), rel * ref.abs() + 1e-45)
            assert r <= 1.0, (depth_mode, r)
            worst = max(worst, r)
        if nch == 4 and conf_mode:
            cref = _conf_ref(shuf[..., 3], conf_mode, cmin, cmax)
            rc = _ratio((conf.double() - cref).abs(), 8 * ULP32 * (cref.abs() + abs(cmin)))
            assert rc <= 1.0, (depth_mode, conf_mode, rc)
            worst = max(worst, rc)
        elif nch == 4:
            assert torch.isnan(conf).all()
    print(f'linear head nch={nch}: worst ratio {worst:.3e}')
