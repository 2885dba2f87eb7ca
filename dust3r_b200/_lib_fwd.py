"""ctypes mirror of the forward-path part of include/dust3r_b200.h ("Path 1")."""
import ctypes as C

F_BIAS, F_GELU, F_RELU, F_OUT_F32, F_RESID_INPLACE = 1, 2, 4, 8, 16
F_ADD0, F_ADD1, F_OUT2_RELU, F_ROPE, F_OUT2_BF16 = 32, 64, 128, 256, 2048


class Linear(C.Structure):
    _fields_ = [('w', C.c_void_p), ('b', C.c_void_p)]


class Norm(C.Structure):
    _fields_ = [('g', C.c_void_p), ('b', C.c_void_p)]


class EncBlock(C.Structure):
    _fields_ = [('norm1', Norm), ('norm2', Norm), ('qkv', Linear), ('proj', Linear), ('fc1', Linear), ('fc2', Linear)]


class DecBlock(C.Structure):
    _fields_ = [('norm1', Norm), ('norm2', Norm), ('norm3', Norm), ('norm_y', Norm),
                ('qkv', Linear), ('proj', Linear), ('projq', Linear), ('projkv', Linear), ('cproj', Linear),
                ('fc1', Linear), ('fc2', Linear)]


class Fusion(C.Structure):
    _fields_ = [('rcu1_conv1', Linear), ('rcu1_conv2', Linear), ('rcu2_conv1', Linear), ('rcu2_conv2', Linear),
                ('out_conv', Linear)]


class DptHead(C.Structure):
    _fields_ = [('act_conv', Linear * 4), ('act0_up', Linear), ('act1_up', Linear), ('act3_down', Linear),
                ('layer_rn', Linear * 4), ('refine', Fusion * 4), ('head0', Linear), ('head2', Linear),
                ('head4_w', C.c_void_p), ('head4_b', C.c_void_p)]


class Model(C.Structure):
    _fields_ = [('enc_dim', C.c_int32), ('enc_depth', C.c_int32), ('enc_heads', C.c_int32), ('dec_dim', C.c_int32),
                ('dec_depth', C.c_int32), ('dec_heads', C.c_int32), ('mlp_ratio', C.c_int32), ('patch', C.c_int32),
                ('head_type', C.c_int32), ('nch', C.c_int32), ('depth_mode', C.c_int32), ('conf_mode', C.c_int32),
                ('conf_min', C.c_float), ('conf_max', C.c_float), ('ln_eps', C.c_float),
                ('hooks', C.c_int32 * 4), ('rope_max_pos', C.c_int32),
                ('rope_cos', C.c_void_p), ('rope_sin', C.c_void_p),
                ('patch_embed', Linear), ('enc', C.POINTER(EncBlock)), ('enc_norm', Norm), ('decoder_embed', Linear),
                ('dec1', C.POINTER(DecBlock)), ('dec2', C.POINTER(DecBlock)), ('dec_norm', Norm),
                ('dpt', C.POINTER(DptHead) * 2), ('lin_head', Linear * 2)]


def declare(lib):
    vp, i32, i64, u32, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_float
    lib.d3r_gemm_bf16.restype = C.c_int
    lib.d3r_gemm_bf16.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i64, u32, vp, vp, i32, i32, i32, vp]
    lib.d3r_conv3x3_bf16.restype = C.c_int
    lib.d3r_conv3x3_bf16.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, u32, vp]
    lib.d3r_attention_hd64.restype = C.c_int
    lib.d3r_attention_hd64.argtypes = [vp, i64, vp, i64, vp, i64, vp, i64, i32, i32, i32, i32, f32, vp]
    lib.d3r_convT_bf16.restype = C.c_int
    lib.d3r_convT_bf16.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.d3r_conv3x3_head_tail.restype = C.c_int
    lib.d3r_conv3x3_head_tail.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, f32, vp]
    lib.d3r_layernorm_bf16.restype = C.c_int
    lib.d3r_layernorm_bf16.argtypes = [vp, vp, vp, vp, i32, i32, f32, vp]
    lib.d3r_upsample2x_bf16.restype = C.c_int
    lib.d3r_upsample2x_bf16.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.d3r_im2col_3x3_s2_bf16.restype = C.c_int
    lib.d3r_im2col_3x3_s2_bf16.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    lib.d3r_patch_im2col16.restype = C.c_int
    lib.d3r_patch_im2col16.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.d3r_gather_images_bf16.restype = C.c_int
    lib.d3r_gather_images_bf16.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.d3r_cast_f32_bf16.restype = C.c_int
    lib.d3r_cast_f32_bf16.argtypes = [vp, vp, i64, vp]
    lib.d3r_linear_head_postprocess.restype = C.c_int
    lib.d3r_linear_head_postprocess.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, f32, f32, vp]
    lib.d3r_set_gemm_impl.restype = None
    lib.d3r_set_gemm_impl.argtypes = [i32]
    lib.d3r_set_attention_impl.restype = None
    lib.d3r_set_attention_impl.argtypes = [i32]
    lib.d3r_forward_workspace_bytes.restype = i64
    lib.d3r_forward_workspace_bytes.argtypes = [C.POINTER(Model), i32, i32, i32, i32]
    lib.d3r_forward_pairs.restype = C.c_int
    lib.d3r_forward_pairs.argtypes = [C.POINTER(Model), vp, i32, C.POINTER(i32), C.POINTER(i32), i32, i32, i32,
                                      vp, vp, vp, vp, vp, i64, vp]
    lib.d3r_forward_mixed_workspace_bytes.restype = i64
    lib.d3r_forward_mixed_workspace_bytes.argtypes = [C.POINTER(Model), i32, i32, i32, i32, i32]
    lib.d3r_forward_pairs_mixed.restype = C.c_int
    lib.d3r_forward_pairs_mixed.argtypes = [C.POINTER(Model), vp, i32, i32, vp, i32, i32, i32, vp, vp, vp, vp, vp, i64, vp]
    lib.d3r_forward_set_debug.restype = C.c_int
    lib.d3r_forward_set_debug.argtypes = [i32, vp, i64]
    lib.d3r_sizeof_model.restype = C.c_int
