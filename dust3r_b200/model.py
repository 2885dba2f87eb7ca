"""AsymmetricCroCo3DStereo — drop-in for dust3r/model.py:46-211 whose forward runs on the B200-native CUDA
path (csrc/forward.cu) through the C ABI.

The module owns fp32 `nn.Parameter`s under the reference's state-dict names (config.state_dict_spec), so
`load_state_dict` / `from_pretrained` accept real DUSt3R checkpoints.  Before the first forward (and after
any weight change) the parameters are repacked once into the kernels' operand layout (bf16 K-major GEMM
weights, tap-major 3x3 filters, fused k|v projection, fp32 biases / LayerNorm parameters, RoPE tables).
There is no torch / CPU fallback: forward() requires a CUDA sm_100 device and the built extension.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from copy import deepcopy

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib_fwd import Model as CModel, EncBlock, DecBlock, DptHead, Fusion, Linear as CLinear, Norm as CNorm
from .config import ModelConfig, state_dict_spec
from .utils.misc import is_symmetrized

inf = float('inf')

try:  # same optional mixin as the reference (model.py:46-52); never needed offline
    import huggingface_hub
    _HubMixin = huggingface_hub.PyTorchModelHubMixin
    _hub_kwargs = dict(library_name="dust3r", repo_url="https://github.com/naver/dust3r", tags=["image-to-3d"])
except Exception:  # pragma: no cover
    class _HubMixin:
        def __init_subclass__(cls, **kw):
            super().__init_subclass__()
    _hub_kwargs = {}


def load_model(model_path, device, verbose=True):
    """dust3r/model.py:27-43: rebuild the network from the constructor string stored in the checkpoint."""
    if verbose:
        print('... loading model from', model_path)
    ckpt = torch.load(model_path, map_location='cpu', weights_only=False)
    args = ckpt['args'].model.replace("ManyAR_PatchEmbed", "PatchEmbedDust3R")
    if 'landscape_only' not in args:
        args = args[:-1] + ', landscape_only=False)'
    else:
        args = args.replace(" ", "").replace('landscape_only=True', 'landscape_only=False')
    assert "landscape_only=False" in args
    if verbose:
        print(f"instantiating : {args}")
    net = eval(args, {'AsymmetricCroCo3DStereo': AsymmetricCroCo3DStereo, 'inf': inf})
    s = net.load_state_dict(ckpt['model'], strict=False)
    if verbose:
        print(s)
    return net.to(device)


def _register(root: nn.Module, dotted: str, param: nn.Parameter):
    """Create (or reuse) the nested containers for `a.b.0.weight` and attach the parameter."""
    parts = dotted.split('.')
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, nn.Module())
        mod = mod._modules[p]
    mod.register_parameter(parts[-1], param)


class AsymmetricCroCo3DStereo(nn.Module, _HubMixin, **_hub_kwargs):
    """Two siamese ViT encoders + two cross-attending decoders + pointmap heads; both pointmaps are
    expressed in view1's frame.  Constructor arguments as in the reference (model.py:58-74,
    croco/models/croco.py:24-37)."""

    def __init__(self, output_mode='pts3d', head_type='linear', depth_mode=('exp', -inf, inf),
                 conf_mode=('exp', 1, inf), freeze='none', landscape_only=True, patch_embed_cls='PatchEmbedDust3R',
                 img_size=224, patch_size=16, mask_ratio=0.9, enc_embed_dim=768, enc_depth=12, enc_num_heads=12,
                 dec_embed_dim=512, dec_depth=8, dec_num_heads=16, mlp_ratio=4, norm_layer=None,
                 norm_im2_in_dec=True, pos_embed='cosine'):
        super().__init__()
        if isinstance(img_size, int):
            img_size = (img_size, img_size)
        assert patch_embed_cls in ['PatchEmbedDust3R', 'ManyAR_PatchEmbed']
        assert img_size[0] % patch_size == 0 and img_size[1] % patch_size == 0, \
            f'{img_size=} must be multiple of {patch_size=}'
        if not pos_embed.startswith('RoPE'):
            raise NotImplementedError('the DUSt3R hot path uses RoPE positional embedding (pos_embed="RoPE100")')
        if output_mode != 'pts3d' or head_type not in ('linear', 'dpt'):
            raise NotImplementedError(f"unexpected {head_type=} and {output_mode=}")
        self.cfg = ModelConfig(img_size=tuple(img_size), patch_size=patch_size, enc_embed_dim=enc_embed_dim,
                               enc_depth=enc_depth, enc_num_heads=enc_num_heads, dec_embed_dim=dec_embed_dim,
                               dec_depth=dec_depth, dec_num_heads=dec_num_heads, mlp_ratio=mlp_ratio, pos_embed=pos_embed,
                               head_type=head_type, output_mode=output_mode, depth_mode=tuple(depth_mode),
                               conf_mode=tuple(conf_mode) if conf_mode else None, landscape_only=landscape_only,
                               norm_im2_in_dec=norm_im2_in_dec)
        if head_type == 'dpt':
            assert dec_depth > 9
        self.patch_embed_cls = patch_embed_cls
        self.croco_args = dict(img_size=img_size, patch_size=patch_size, mask_ratio=mask_ratio, enc_embed_dim=enc_embed_dim,
                               enc_depth=enc_depth, enc_num_heads=enc_num_heads, dec_embed_dim=dec_embed_dim,
                               dec_depth=dec_depth, dec_num_heads=dec_num_heads, mlp_ratio=mlp_ratio,
                               norm_im2_in_dec=norm_im2_in_dec, pos_embed=pos_embed)
        self.patch_size = patch_size
        self.enc_depth, self.enc_embed_dim = enc_depth, enc_embed_dim
        self.dec_depth, self.dec_embed_dim = dec_depth, dec_embed_dim
        self.output_mode, self.head_type = output_mode, head_type
        self.depth_mode, self.conf_mode = depth_mode, conf_mode
        self.pos_embed = pos_embed
        self.landscape_only = landscape_only

        spec = state_dict_spec(self.cfg)
        made = {}
        for key, shape in spec.items():
            if '.scratch.layer_rn.' in key:   # alias of scratch.layer{k+1}_rn (same storage, dpt_block.py:72-77)
                k = int(key.split('.scratch.layer_rn.')[1].split('.')[0])
                src = key.replace(f'.scratch.layer_rn.{k}.', f'.scratch.layer{k + 1}_rn.')
                _register(self, key, made[src])
                continue
            p = nn.Parameter(self._init_tensor(key, shape))
            made[key] = p
            _register(self, key, p)
        self.set_freeze(freeze)
        self._packed = None
        self.eval()

    # ---------------------------------------------------------------- init / loading
    @staticmethod
    def _init_tensor(key, shape):
        """croco.py:111-127: xavier-uniform linears, zero biases, unit LayerNorms, N(0,0.02) mask token;
        convolutions keep torch's default (kaiming-uniform(a=sqrt(5)))."""
        t = torch.empty(shape)
        if key == 'mask_token':
            return nn.init.normal_(t, std=.02)
        if key.endswith('bias'):
            if len(shape) == 1 and ('.dpt.' in key):
                return nn.init.uniform_(t, -0.05, 0.05)
            return nn.init.zeros_(t)
        if '.norm' in key or key.startswith(('enc_norm', 'dec_norm')):
            return nn.init.ones_(t)
        if len(shape) == 2:
            return nn.init.xavier_uniform_(t)
        if key == 'patch_embed.proj.weight':
            nn.init.xavier_uniform_(t.view(shape[0], -1))
            return t
        return nn.init.kaiming_uniform_(t, a=math.sqrt(5))

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, **kw):
        if os.path.isfile(pretrained_model_name_or_path):
            return load_model(pretrained_model_name_or_path, device='cpu')
        try:
            return super(AsymmetricCroCo3DStereo, cls).from_pretrained(pretrained_model_name_or_path, **kw)
        except TypeError as e:
            raise Exception(f'tried to load {pretrained_model_name_or_path} from huggingface, but failed') from e

    def load_state_dict(self, ckpt, **kw):
        new_ckpt = dict(ckpt)
        if not any(k.startswith('dec_blocks2') for k in ckpt):   # model.py:91-98
            for key, value in ckpt.items():
                if key.startswith('dec_blocks'):
                    new_ckpt[key.replace('dec_blocks', 'dec_blocks2')] = value
        self._packed = None
        return super().load_state_dict(new_ckpt, **kw)

    def _apply(self, fn, *a, **kw):
        self._packed = None
        return super()._apply(fn, *a, **kw)

    def set_freeze(self, freeze):
        self.freeze = freeze
        assert freeze in ('none', 'mask', 'encoder')
        if freeze in ('mask', 'encoder'):
            self.mask_token.requires_grad = False
        if freeze == 'encoder':
            for n, p in self.named_parameters():
                if n.startswith(('patch_embed.', 'enc_blocks.')):
                    p.requires_grad = False

    # ---------------------------------------------------------------- weight repacking
    def _param_version(self):
        """Sum of the parameters' in-place modification counters: changes whenever a weight is edited in place
        (p.data.copy_, optimizer steps, ...), which load_state_dict / .to() hooks cannot see."""
        return sum(p._version for p in self.parameters())

    def repack(self):
        """(Re)build the kernel-side operand buffers (bf16 GEMM operands, fp32 biases / LayerNorm parameters) from the
        current parameters.  forward() calls it by itself when the parameters changed since the last packing."""
        dev = next(self.parameters()).device
        _lib.require_cuda_device(dev)
        self._packed = _PackedModel(self, dev)
        self._packed_version = self._param_version()
        return self._packed

    def _ensure_packed(self, dev):
        if self._packed is None or self._packed.device != dev or getattr(self, '_packed_version', None) != self._param_version():
            if next(self.parameters()).device != dev:
                raise _lib.D3RError(f'model parameters live on {next(self.parameters()).device}, images on {dev}')
            self.repack()

    # ---------------------------------------------------------------- forward
    @torch.no_grad()
    def forward(self, view1, view2):
        img1, img2 = view1['img'], view2['img']
        B = img1.shape[0]
        dev = img1.device
        _lib.require_cuda_device(dev)
        self._ensure_packed(dev)
        H, W = int(img1.shape[-2]), int(img1.shape[-1])
        H2, W2 = int(img2.shape[-2]), int(img2.shape[-1])
        shape1 = torch.as_tensor(view1.get('true_shape', torch.tensor(img1.shape[-2:])[None].repeat(B, 1))).cpu()
        shape2 = torch.as_tensor(view2.get('true_shape', torch.tensor(img2.shape[-2:])[None].repeat(B, 1))).cpu()
        if self.landscape_only:
            # ManyAR batches (patch_embed.py:32-70 + transpose_to_landscape.wrapper_yes, utils/misc.py:66-95): every image
            # tensor is stored in landscape; items whose true_shape says portrait are the transposed storage of a portrait image
            port1, port2 = shape1[:, 0] > shape1[:, 1], shape2[:, 0] > shape2[:, 1]
            for ts, port, (Hv, Wv) in ((shape1, port1, (H, W)), (shape2, port2, (H2, W2))):
                assert Wv >= Hv, f'img should be in landscape mode, but got W={Wv} H={Hv}'
                want = torch.where(port[:, None], torch.tensor([[Wv, Hv]]), torch.tensor([[Hv, Wv]]))
                assert bool((ts == want).all()), 'true_shape must be the image tensor size (landscape) or its transpose (portrait)'
            if bool(port1.any()) or bool(port2.any()):
                return self._forward_many_ar(view1, view2, port1, port2)
        for ts, (Hv, Wv) in ((shape1, (H, W)), (shape2, (H2, W2))):
            assert ts[0:1].allclose(ts), 'true_shape must be all identical'
            h, w = [int(v) for v in ts[0].tolist()]
            if (h, w) != (Hv, Wv):
                raise AssertionError(f'true_shape {(h, w)} does not match the image tensor {(Hv, Wv)}')
        if (H, W) != (H2, W2):
            # model.py:147-151: the two views are encoded separately; the decoder cross-attends between the two grids
            res1, res2 = self._packed.forward_mixed(img1.float().contiguous(), img2.float().contiguous())
            res2['pts3d_in_other_view'] = res2.pop('pts3d')
            return res1, res2
        # model.py:153-170: a batch [(a,b),(b,a),...] only encodes its even half
        if is_symmetrized(view1, view2):
            imgs = torch.cat((img1[::2], img2[::2]), dim=0)
            half = B // 2
            idx1 = np.empty(B, dtype=np.int32)
            idx2 = np.empty(B, dtype=np.int32)
            idx1[0::2] = np.arange(half); idx1[1::2] = half + np.arange(half)
            idx2[0::2] = half + np.arange(half); idx2[1::2] = np.arange(half)
        else:
            imgs = torch.cat((img1, img2), dim=0)
            idx1 = np.arange(B, dtype=np.int32)
            idx2 = B + np.arange(B, dtype=np.int32)
        res1, res2 = self._packed.forward(imgs.float().contiguous(), idx1, idx2, B, H, W)
        res2['pts3d_in_other_view'] = res2.pop('pts3d')
        return res1, res2


    def _forward_many_ar(self, view1, view2, port1, port2):
        """landscape_only=True with portrait items: the reference embeds a portrait item from its un-transposed pixels
        (ManyAR_PatchEmbed), runs the head at the portrait size and transposes the result back (wrapper_yes) -- per image
        that is exactly transpose(model(un-transposed image)).  Items are grouped by the orientation of their two views (at
        most four groups); each group is an ordinary batch (a landscape/portrait pair is a pair of two image sizes)."""
        img1, img2 = view1['img'], view2['img']
        B = img1.shape[0]
        out1, out2 = {}, {}
        for p1 in (False, True):
            for p2 in (False, True):
                sel = torch.nonzero((port1 == p1) & (port2 == p2)).flatten()
                if sel.numel() == 0:
                    continue
                seld = sel.to(img1.device)
                a, b = img1.index_select(0, seld), img2.index_select(0, seld)
                a = a.swapaxes(-1, -2).contiguous() if p1 else a
                b = b.swapaxes(-1, -2).contiguous() if p2 else b
                was, self.landscape_only = self.landscape_only, False
                try:
                    n = int(sel.numel())   # distinct instance names: no symmetrised-batch shortcut inside a group (same results)
                    r1, r2 = self.forward(dict(img=a, instance=[f'a{i}' for i in range(n)]), dict(img=b, instance=[f'b{i}' for i in range(n)]))
                finally:
                    self.landscape_only = was
                for res, port, out in ((r1, p1, out1), (r2, p2, out2)):
                    for k, v in res.items():
                        v = v.swapaxes(1, 2) if port else v
                        if k not in out:
                            out[k] = v.new_empty((B,) + tuple(v.shape[1:]))
                        out[k].index_copy_(0, seld, v.contiguous())
        return out1, out2

    def forward_indexed(self, imgs, idx1, idx2):
        """Extension used by inference(): `imgs` (n,3,H,W) are the DISTINCT images of a batch (CUDA), pair b is
        (imgs[idx1[b]], imgs[idx2[b]]).  The encoder runs once per distinct image (the reference encodes every pair's
        two images again, model.py:142-170; a symmetrised batch is the special case it shortcuts); decoder and heads
        run per pair.  Same outputs as forward() on the expanded batch."""
        dev = imgs.device
        _lib.require_cuda_device(dev)
        self._ensure_packed(dev)
        B = len(idx1)
        assert len(idx2) == B and B > 0
        H, W = int(imgs.shape[-2]), int(imgs.shape[-1])
        res1, res2 = self._packed.forward(imgs.float().contiguous(), np.asarray(idx1, dtype=np.int32), np.asarray(idx2, dtype=np.int32), B, H, W)
        res2['pts3d_in_other_view'] = res2.pop('pts3d')
        return res1, res2


def pack_conv3x3(w):
    """(Cout, Cin, 3, 3) Conv2d weight -> [Cout][ky][kx][Cin]: the B operand of the implicit-GEMM 3x3 conv."""
    return w.permute(0, 2, 3, 1).contiguous()


def pack_conv3x3_s2(w):
    """(Cout, Cin, 3, 3) Conv2d weight -> [Cout][(ky*3+kx)*Cin + ci]: the GEMM operand over d3r_im2col_3x3_s2_bf16 rows."""
    return pack_conv3x3(w).reshape(w.shape[0], -1)


def pack_convT(w):
    """(Cin, Cout, k, k) ConvTranspose2d weight (k == stride) -> [(ky*k+kx)*Cout + co][ci]: the B operand of d3r_convT_bf16."""
    ci, co, k, _ = w.shape
    return w.permute(2, 3, 1, 0).reshape(k * k * co, ci).contiguous()


class _PackedModel:
    """Device-side operand buffers + the ctypes `d3r_model` descriptor pointing at them."""

    def __init__(self, net: AsymmetricCroCo3DStereo, device):
        self.device = device
        self.cfg = cfg = net.cfg
        self.lib = _lib.get_lib()
        self._keep = []      # tensors referenced by raw pointers
        sd = {k: v.detach() for k, v in net.state_dict().items()}
        E, D = cfg.enc_embed_dim, cfg.dec_embed_dim

        def bf(t):
            t = t.to(device=device, dtype=torch.bfloat16).contiguous()
            self._keep.append(t)
            return t.data_ptr()

        def f32(t):
            t = t.to(device=device, dtype=torch.float32).contiguous()
            self._keep.append(t)
            return t.data_ptr()

        def lin(prefix, w=None, b='auto'):
            w = sd[prefix + '.weight'] if w is None else w
            bias = sd.get(prefix + '.bias') if isinstance(b, str) else b
            return CLinear(bf(w.reshape(w.shape[0], -1)), f32(bias) if bias is not None else None)

        def norm(prefix):
            return CNorm(f32(sd[prefix + '.weight']), f32(sd[prefix + '.bias']))

        def conv3(prefix):
            bias = sd.get(prefix + '.bias')
            return CLinear(bf(pack_conv3x3(sd[prefix + '.weight'])), f32(bias) if bias is not None else None)

        def convT(prefix):
            return CLinear(bf(pack_convT(sd[prefix + '.weight'])), f32(sd[prefix + '.bias']))

        m = CModel()
        m.enc_dim, m.enc_depth, m.enc_heads = E, cfg.enc_depth, cfg.enc_num_heads
        m.dec_dim, m.dec_depth, m.dec_heads = D, cfg.dec_depth, cfg.dec_num_heads
        m.mlp_ratio, m.patch = int(cfg.mlp_ratio), cfg.patch_size
        m.head_type = 1 if cfg.head_type == 'dpt' else 0
        m.nch = 3 + int(cfg.has_conf)
        dmode = cfg.depth_mode[0]
        assert cfg.depth_mode[1] == -inf and cfg.depth_mode[2] == inf, 'bounded depth modes are not used by DUSt3R'
        m.depth_mode = {'linear': 0, 'square': 1, 'exp': 2}[dmode]
        if cfg.conf_mode:
            m.conf_mode = {'exp': 1, 'sigmoid': 2}[cfg.conf_mode[0]]
            m.conf_min = float(cfg.conf_mode[1])
            m.conf_max = float(min(cfg.conf_mode[2], 3.0e38))
        else:
            m.conf_mode, m.conf_min, m.conf_max = 0, 0.0, 0.0
        m.ln_eps = 1e-6
        # RoPE tables: angle[p][k] = p * base^(-k/16)   (croco/models/curope/kernels.cu:41-52, hd = 64)
        max_pos = max(64, max(cfg.img_size) // cfg.patch_size * 2)
        inv_freq = 1.0 / (cfg.rope_freq ** (torch.arange(0, 16).float() / 16))
        ang = torch.arange(max_pos).float()[:, None] * inv_freq[None, :]
        m.rope_max_pos = max_pos
        m.rope_cos, m.rope_sin = f32(ang.cos()), f32(ang.sin())
        m.patch_embed = lin('patch_embed.proj')
        self._enc = (EncBlock * cfg.enc_depth)()
        for i in range(cfg.enc_depth):
            p = f'enc_blocks.{i}'
            b = self._enc[i]
            b.norm1, b.norm2 = norm(p + '.norm1'), norm(p + '.norm2')
            b.qkv, b.proj = lin(p + '.attn.qkv'), lin(p + '.attn.proj')
            b.fc1, b.fc2 = lin(p + '.mlp.fc1'), lin(p + '.mlp.fc2')
        m.enc = C.cast(self._enc, C.POINTER(EncBlock))
        m.enc_norm = norm('enc_norm')
        m.decoder_embed = lin('decoder_embed')
        self._dec = []
        for name in ('dec_blocks', 'dec_blocks2'):
            arr = (DecBlock * cfg.dec_depth)()
            for i in range(cfg.dec_depth):
                p = f'{name}.{i}'
                b = arr[i]
                b.norm1, b.norm2, b.norm3 = norm(p + '.norm1'), norm(p + '.norm2'), norm(p + '.norm3')
                if not cfg.norm_im2_in_dec:
                    raise NotImplementedError('norm_im2_in_dec=False (identity memory norm) is not used by DUSt3R')
                b.norm_y = norm(p + '.norm_y')
                b.qkv, b.proj = lin(p + '.attn.qkv'), lin(p + '.attn.proj')
                b.projq = lin(p + '.cross_attn.projq')
                wkv = torch.cat((sd[p + '.cross_attn.projk.weight'], sd[p + '.cross_attn.projv.weight']), dim=0)
                bkv = torch.cat((sd[p + '.cross_attn.projk.bias'], sd[p + '.cross_attn.projv.bias']), dim=0)
                b.projkv = lin(None, w=wkv, b=bkv)
                b.cproj = lin(p + '.cross_attn.proj')
                b.fc1, b.fc2 = lin(p + '.mlp.fc1'), lin(p + '.mlp.fc2')
            self._dec.append(arr)
        m.dec1 = C.cast(self._dec[0], C.POINTER(DecBlock))
        m.dec2 = C.cast(self._dec[1], C.POINTER(DecBlock))
        m.dec_norm = norm('dec_norm')
        self._dpt = []
        if cfg.head_type == 'dpt':
            assert cfg.norm_im2_in_dec
            for k, h in enumerate(cfg.dpt_hooks):
                m.hooks[k] = h
            for hnum in (1, 2):
                p = f'downstream_head{hnum}.dpt'
                hd = DptHead()
                for k in range(4):
                    hd.act_conv[k] = lin(f'{p}.act_postprocess.{k}.0')
                    hd.layer_rn[k] = conv3(f'{p}.scratch.layer{k + 1}_rn')
                hd.act0_up = convT(f'{p}.act_postprocess.0.1')
                hd.act1_up = convT(f'{p}.act_postprocess.1.1')
                hd.act3_down = lin(None, w=pack_conv3x3_s2(sd[f'{p}.act_postprocess.3.1.weight']),
                                   b=sd[f'{p}.act_postprocess.3.1.bias'])
                for r in range(4):
                    q = f'{p}.scratch.refinenet{r + 1}'
                    f = hd.refine[r]
                    f.rcu1_conv1, f.rcu1_conv2 = conv3(q + '.resConfUnit1.conv1'), conv3(q + '.resConfUnit1.conv2')
                    f.rcu2_conv1, f.rcu2_conv2 = conv3(q + '.resConfUnit2.conv1'), conv3(q + '.resConfUnit2.conv2')
                    f.out_conv = lin(q + '.out_conv')
                hd.head0, hd.head2 = conv3(p + '.head.0'), conv3(p + '.head.2')
                w4 = torch.zeros((4, 128))          # kernel reads 4 rows; row 3 stays zero without confidence
                w4[:m.nch] = sd[p + '.head.4.weight'].reshape(m.nch, -1).float().cpu()
                b4 = torch.zeros((4,))
                b4[:m.nch] = sd[p + '.head.4.bias'].float().cpu()
                hd.head4_w, hd.head4_b = f32(w4), f32(b4)
                self._dpt.append(hd)
                m.dpt[hnum - 1] = C.pointer(hd)
        else:
            m.lin_head[0] = lin('downstream_head1.proj')
            m.lin_head[1] = lin('downstream_head2.proj')
        self.cmodel = m
        self._ws = None
        self._ws_key = None

    def workspace(self, n_enc, B, H, W):
        key = (n_enc, B, H, W)
        if self._ws_key != key:
            need = self.lib.d3r_forward_workspace_bytes(C.byref(self.cmodel), n_enc, B, H, W)
            if need <= 0:
                _lib.check(-1)
            self._ws = None   # free the old one first
            self._ws = torch.empty((need,), dtype=torch.uint8, device=self.device)
            self._ws_key = key
        return self._ws

    def forward_mixed(self, imgs1, imgs2):
        """imgs1 (B,3,H1,W1), imgs2 (B,3,H2,W2) fp32 CUDA with different sizes -> ({'pts3d','conf'}, {'pts3d','conf'})."""
        B = int(imgs1.shape[0])
        assert int(imgs2.shape[0]) == B
        H1, W1, H2, W2 = int(imgs1.shape[-2]), int(imgs1.shape[-1]), int(imgs2.shape[-2]), int(imgs2.shape[-1])
        key = ('mixed', B, H1, W1, H2, W2)
        if self._ws_key != key:
            need = self.lib.d3r_forward_mixed_workspace_bytes(C.byref(self.cmodel), B, H1, W1, H2, W2)
            if need <= 0:
                _lib.check(-1)
            self._ws = None
            self._ws = torch.empty((need,), dtype=torch.uint8, device=self.device)
            self._ws_key = key
        dev = self.device
        has_conf = self.cmodel.nch > 3
        pts1 = torch.empty((B, H1, W1, 3), dtype=torch.float32, device=dev)
        pts2 = torch.empty((B, H2, W2, 3), dtype=torch.float32, device=dev)
        conf1 = torch.empty((B, H1, W1), dtype=torch.float32, device=dev) if has_conf else None
        conf2 = torch.empty((B, H2, W2), dtype=torch.float32, device=dev) if has_conf else None
        with torch.cuda.device(dev):
            _lib.check(self.lib.d3r_forward_pairs_mixed(C.byref(self.cmodel), imgs1.data_ptr(), H1, W1, imgs2.data_ptr(), H2, W2, B,
                                                        pts1.data_ptr(), conf1.data_ptr() if has_conf else None,
                                                        pts2.data_ptr(), conf2.data_ptr() if has_conf else None,
                                                        self._ws.data_ptr(), self._ws.numel(), _lib.stream_ptr()))
        r1, r2 = {'pts3d': pts1}, {'pts3d': pts2}
        if has_conf:
            r1['conf'], r2['conf'] = conf1, conf2
        return r1, r2

    def forward(self, imgs, idx1, idx2, B, H, W, debug=None):
        """imgs: (n_enc,3,H,W) fp32 CUDA.  Returns ({'pts3d','conf'}, {'pts3d','conf'}) CUDA fp32 tensors."""
        n_enc = int(imgs.shape[0])
        ws = self.workspace(n_enc, B, H, W)
        dev = self.device
        has_conf = self.cmodel.nch > 3
        pts1 = torch.empty((B, H, W, 3), dtype=torch.float32, device=dev)
        pts2 = torch.empty((B, H, W, 3), dtype=torch.float32, device=dev)
        conf1 = torch.empty((B, H, W), dtype=torch.float32, device=dev) if has_conf else None
        conf2 = torch.empty((B, H, W), dtype=torch.float32, device=dev) if has_conf else None
        i1 = (C.c_int32 * B)(*[int(v) for v in idx1])
        i2 = (C.c_int32 * B)(*[int(v) for v in idx2])
        if debug is not None:
            stage, buf = debug
            _lib.check(self.lib.d3r_forward_set_debug(stage, buf.data_ptr(), buf.numel()))
        with torch.cuda.device(dev):
            _lib.check(self.lib.d3r_forward_pairs(C.byref(self.cmodel), imgs.data_ptr(), n_enc, i1, i2, B, H, W,
                                                  pts1.data_ptr(), conf1.data_ptr() if has_conf else None,
                                                  pts2.data_ptr(), conf2.data_ptr() if has_conf else None,
                                                  ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
        r1, r2 = {'pts3d': pts1}, {'pts3d': pts2}
        if has_conf:
            r1['conf'], r2['conf'] = conf1, conf2
        return r1, r2
