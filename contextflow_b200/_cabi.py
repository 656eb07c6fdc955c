"""ctypes binding of libcfpp.so (include/cfpp.h).  There is no CPU fallback: a missing library is a hard error."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('CFPP_LIB') or os.path.join(_HERE, 'libcfpp.so')   # CFPP_LIB: an experimental build of the same sources (tools/ A/B runs)

MAX_CTX = 8
ENC_MAXC = 64
MAX_ENC_BATCH = 64
EMB = dict(onehot=0, eye=1, embed=2, dense=3)
ENC = dict(eyesample=0, uniform=1, vardeq=2, argmax=3, probsample=4)

vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float


class VitDesc(C.Structure):
    _fields_ = [('Cin', i32), ('H', i32), ('W', i32), ('p1', i32), ('p2', i32),
                ('T', i32), ('depth', i32), ('n_tok', i32), ('patch_dim', i32),
                ('ln0_w', vp), ('ln0_b', vp), ('pe_wt', vp), ('pe_b', vp), ('ln1_w', vp), ('ln1_b', vp),
                ('pos', vp), ('lnf_w', vp), ('lnf_b', vp), ('layers', vp)]


class EncDesc(C.Structure):
    _fields_ = [('emb', i32), ('type', i32), ('n_ctx', i32), ('C', i32),
                ('card', i32 * MAX_CTX), ('bits', i32 * MAX_CTX), ('emb_dim', i32),
                ('emb_w', vp * MAX_CTX), ('dense', vp), ('qbins', vp), ('ldj_per_dim', vp), ('temperature', vp),
                ('inner_dim', i32), ('inner_w', vp * MAX_CTX),
                ('fc', vp * 2), ('fc_logabsdet', vp * 2), ('an_t', vp * 2), ('an_logs', vp * 2),
                ('cw1t', vp * 2), ('cb1', vp * 2), ('cw2t', vp * 2), ('cb2', vp * 2), ('cw3t', vp * 2), ('cb3', vp * 2)]


class CnJob(C.Structure):
    _fields_ = [('w', vp * 3), ('b', vp * 3), ('n_layers', i32), ('K', i32), ('N', i32 * 3), ('tril_dim', i32)]


MAX_CN_JOBS = 64

_SIGNATURES = {
    'cfpp_version': (i32, []),
    'cfpp_last_error': (C.c_char_p, []),
    'cfpp_launch_count': (i64, []),
    'cfpp_copy_peer_async': (i32, [vp, i32, vp, i32, i64, vp]),
    'cfpp_maf_coupling_ctx_fwd': (i32, [vp, vp, vp, vp, f32, vp, vp, i32, i32, i32, vp]),
    'cfpp_adamw_chunk': (i32, []),
    'cfpp_adamw_step': (i32, [vp, vp, i32, vp, vp, C.c_double, C.c_double, C.c_double, C.c_double, vp]),
    'cfpp_activation_fwd': (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    'cfpp_activation_inv': (i32, [vp, vp, vp, i64, f32, i32, vp]),
    'cfpp_activation_bwd': (i32, [vp, vp, vp, vp, vp, i64, i32, i32, vp]),
    'cfpp_student_table_floats': (i64, [i32, i32, i32]),
    'cfpp_student_prep': (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_student_logprob': (i32, [vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_student_train_fwd': (i32, [vp, i64, vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_student_train_bwd_workspace_floats': (i64, [i32, i32, i32, i32]),
    'cfpp_student_train_bwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_bias_rows_relu': (i32, [vp, vp, i32, i32, i32, vp]),
    'cfpp_gmm_ctx_param_bwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_squeeze_fwd': (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_squeeze_strided_fwd': (i32, [vp, i64, vp, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_squeeze_inv': (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_permute_fwd': (i32, [vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_slice_channels': (i32, [vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_place_channels': (i32, [vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_windows_fwd': (i32, [vp, i32, vp, i64, i64, vp, i32, i64, i32, i32, vp]),
    'cfpp_add_fwd': (i32, [vp, vp, vp, i64, vp]),
    'cfpp_normalize_fwd': (i32, [vp, vp, i64, f32, f32, vp]),
    'cfpp_logit_fwd': (i32, [vp, vp, vp, i32, i32, vp]),
    'cfpp_augment_fwd': (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_prologue_fwd': (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, f32, f32, f32, f32, vp]),
    'cfpp_slogdet': (i32, [vp, i32, vp, vp]),
    'cfpp_conv1x1_fwd': (i32, [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, vp, f32, i32, i32, i32, vp]),
    'cfpp_conv1x1_ctx_supported': (i32, [i32, i32, i32, i32]),
    'cfpp_conv1x1_ctx_fwd': (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, vp, f32, i32, i32, i32, i32, vp]),
    'cfpp_actnorm_fwd': (i32, [vp, vp, vp, vp, vp, vp, vp, f32, i32, i32, i32, i32, vp]),
    'cfpp_actnorm_stats': (i32, [vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_coupling_fwd': (i32, [vp, vp, vp, vp, f32, vp, vp, i32, i32, i32, vp]),
    'cfpp_conv_cond_fwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv_cond_tc_pack_bytes': (i64, [i32, i32, i32, i32, i32]),
    'cfpp_conv_cond_tc_pack': (i32, [vp, i32, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv_cond_tc_supported': (i32, [i32, i32, i32, i32, i32, i32, i32, i32, i64]),
    'cfpp_conv_cond_tc_fwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv_cond_tc_train_fwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv_cond_tc_coupling_supported': (i32, [i32, i32, i32, i32, i32, i32, i32]),
    'cfpp_conv_cond_tc_coupling_fwd': (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, f32, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv_cond_tc_kind': (i32, []),
    'cfpp_conv_cond_tc_last_plan': (None, [C.POINTER(i32)]),
    'cfpp_conv_cond_tc_set_profile': (None, [vp]),
    'cfpp_vit_layer_floats': (i64, [i32]),
    'cfpp_vit_cond_fwd': (i32, [vp, i64, vp, i32, vp, C.POINTER(VitDesc), i32, vp]),
    'cfpp_vit_tc_supported': (i32, [i32, i32, i32, i32]),
    'cfpp_vit_tc_pack_bytes': (i64, [i32]),
    'cfpp_vit_tc_pack_chunk': (i32, [vp, i32, i32, i32, vp, vp]),
    'cfpp_vit_tc_fwd': (i32, [vp, i64, vp, C.POINTER(VitDesc), vp, i32, vp]),
    'cfpp_vit_tc2_supported': (i32, [i32, i32, i32, i32]),
    'cfpp_vit_tc2_chunks': (i64, [i32, i32, i32]),
    'cfpp_vit_tc2_fwd': (i32, [vp, i64, vp, C.POINTER(VitDesc), vp, i32, vp]),
    'cfpp_gmm_logprob': (i32, [vp, i64, vp, vp, vp, vp, vp, f32, vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_gmm_logprob_ctxtab': (i32, [vp, i64, vp, vp, vp, vp, i32, C.POINTER(i32), C.POINTER(vp), i32, vp, f32, vp, vp, i64,
                                      i32, i32, i32, i32, i32, vp]),
    'cfpp_gmm_logprob_ctxtab_cached': (i32, [vp, i64, vp, vp, vp, vp, i32, C.POINTER(i32), C.POINTER(vp), i32, vp, f32, vp, vp, i64,
                                             i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_gmm_ctxtab_workspace_bytes': (i64, [i32, i32, i32, i32, i32, i32, C.POINTER(i32)]),
    'cfpp_gmm_workspace_floats': (i64, [i32, i32, i32, i32]),
    'cfpp_gmm_tile_table_bytes': (i64, [i32, i32, i32, i32, i32]),
    'cfpp_gmm_tile_prepare': (i32, [vp, vp, vp, vp, i32, i32, i32, vp, i32, i32, i32, i32, vp]),
    'cfpp_gmm_tile_workspace_bytes': (i64, [i32, i32, i32, i32, i32, i32]),
    'cfpp_gmm_tile_logprob': (i32, [vp, i64, vp, vp, i32, C.POINTER(i32), vp, i32, i32, vp, f32, vp, vp, i64, i32, i32, i32, i32, i32, vp]),
    'cfpp_ctx_encode': (i32, [vp, vp, vp, vp, C.POINTER(EncDesc), i32, i32, vp]),
    'cfpp_ctx_encode_batch': (i32, [vp, vp, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i32, vp]),
    'cfpp_ctx_encode_flow_supported': (i32, [i32]),
    'cfpp_ctx_encode_batch_flow': (i32, [vp, vp, i32, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i32, vp]),
    'cfpp_embed_lookup': (i32, [vp, C.POINTER(vp), i32, i32, vp, i32, vp]),
    'cfpp_linear_fwd': (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_cn_batch': (i32, [C.POINTER(CnJob), i32, C.POINTER(vp), C.POINTER(vp), i32, vp]),
    'cfpp_relu_fwd': (i32, [vp, vp, i64, vp]),
    'cfpp_maf_coupling_fwd': (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_maf_coupling_bwd': (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_coupling_inv': (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_actnorm_inv': (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_mat_inverse': (i32, [vp, i32, vp, vp, vp]),
    'cfpp_sigmoid_fwd': (i32, [vp, vp, i64, vp]),
    'cfpp_normalize_inv': (i32, [vp, vp, i64, f32, f32, vp]),
    'cfpp_floor_fwd': (i32, [vp, vp, i64, vp]),
    'cfpp_prologue_inv': (i32, [vp, vp, vp, i32, i32, i32, i32, f32, f32, f32, f32, i32, vp]),
    'cfpp_gmm_sample': (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_score_workspace_bytes': (i64, [i32]),
    'cfpp_score_epilogue': (i32, [vp, f32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]),
    'cfpp_coupling_bwd': (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_conv1x1_ctx_bwd': (i32, [vp, vp, vp, vp, i32, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_actnorm_ctx_bwd': (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_actnorm_bwd_workspace_floats': (i64, [i32, i32]),
    'cfpp_actnorm_bwd': (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_conv2d_fwd': (i32, [vp, i64, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv2d_bwd_data': (i32, [vp, vp, vp, i64, vp, i64, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_conv2d_bwd_weight_workspace_floats': (i64, [i32, i32, i32, i32, i32]),
    'cfpp_conv2d_bwd_weight': (i32, [vp, i64, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_relu_mask': (i32, [vp, vp, i64, vp]),
    'cfpp_logdet_grad': (i32, [vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_rowsum': (i32, [vp, vp, i32, i32, vp]),
    'cfpp_gmm_train_prep': (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    'cfpp_gmm_train_fwd': (i32, [vp, i64, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_gmm_train_bwd_workspace_floats': (i64, [i32, i32, i32, i32]),
    'cfpp_gmm_train_bwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    'cfpp_gmm_ctx_train_fwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_gmm_ctx_train_bwd': (i32, [vp, i64, vp, vp, vp, vp, vp, vp, i64, vp, i32, i32, i32, i32, i32, vp]),
    'cfpp_cond_gauss_fwd': (i32, [vp, vp, vp, vp, i32, i32, vp]),
    'cfpp_cond_gauss_bwd': (i32, [vp, vp, vp, vp, vp, i32, i32, vp]),
    'cfpp_vardeq_fwd': (i32, [vp, vp, vp, vp, f32, i32, vp, vp, i32, i32, vp]),
    'cfpp_vardeq_bwd': (i32, [vp, vp, vp, i32, vp, vp, vp, vp, i32, i32, vp]),
    'cfpp_embed_scatter': (i32, [vp, i64, i32, vp, vp, vp, i32, i32, vp]),
    'cfpp_patchify_fwd': (i32, [vp, i64, vp, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_patchify_inv': (i32, [vp, vp, i64, i32, i32, i32, i32, i32, i32, i32, vp]),
    'cfpp_layernorm_fwd': (i32, [vp, vp, vp, vp, vp, vp, i64, i32, vp]),
    'cfpp_layernorm_bwd_workspace_floats': (i64, [i64, i32]),
    'cfpp_layernorm_bwd': (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp]),
    'cfpp_rows_linear_fwd': (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    'cfpp_rows_linear_bwd_data': (i32, [vp, vp, vp, i32, i64, i32, i32, vp]),
    'cfpp_rows_linear_bwd_weight_workspace_floats': (i64, [i64, i32, i32]),
    'cfpp_rows_linear_bwd_weight': (i32, [vp, vp, vp, vp, vp, i64, i32, i32, vp]),
    'cfpp_gelu_fwd': (i32, [vp, vp, i64, vp]),
    'cfpp_gelu_bwd': (i32, [vp, vp, vp, i64, vp]),
    'cfpp_add_pos': (i32, [vp, vp, i64, i32, i32, vp]),
    'cfpp_attention_fwd': (i32, [vp, vp, vp, i32, i32, vp]),
    'cfpp_attention_bwd': (i32, [vp, vp, vp, vp, i32, i32, vp]),
    'cfpp_ldj_accumulate': (i32, [vp, vp, i32, i32, i32, vp]),
    'cfpp_ldj_sum': (i32, [vp, vp, vp, C.POINTER(vp), C.POINTER(i32), i32, i32, i32, vp]),
}

_lib = None


def lib():
    """The loaded CUDA library; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                '(nvcc, sm_100a).  contextflow_b200 has no CPU or PyTorch fallback for its kernels.')
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int, what: str = ''):
    if rc != 0:
        msg = lib().cfpp_last_error().decode(errors='replace')
        raise RuntimeError(f'libcfpp {what} failed (status {rc}): {msg}')


def launch_count() -> int:
    return int(lib().cfpp_launch_count())
