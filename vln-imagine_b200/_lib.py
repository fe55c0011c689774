"""ctypes binding of libvlnimagine.so (include/vlnimagine.h).

The library is the only compute back end: if it is missing or fails to load, importing this
module raises - there is no CPU / eager-PyTorch fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libvlnimagine.so')

if not os.path.exists(LIB_PATH):
    raise ImportError(
        'libvlnimagine.so is not built (expected at %s). Run `python -c "import __graft_entry__ as g; g.build()"` '
        'or `python vln-imagine_b200/build.py`; there is no fallback path.' % LIB_PATH)

lib = C.CDLL(LIB_PATH)

VI_OK = 0
DT_BF16, DT_F32, DT_F16 = 0, 1, 2
LN_NONE, LN_FOLD, LN_RESIDUAL = 0, 1, 2
EPI_NONE, EPI_GELU, EPI_RELU = 0, 1, 2
MASK_ADD_NEG10000, MASK_NEG_INF = 0, 1

_p, _i, _l, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float
_ip = C.POINTER(C.c_int32)


class EmbedArgs(C.Structure):
    _fields_ = [
        ('a', _p), ('a_gamma', _p), ('a_beta', _p),
        ('feat', _p), ('feat_dim', C.c_int32), ('feat_w', _p), ('feat_b', _p), ('feat_gamma', _p), ('feat_beta', _p),
        ('idx', _p), ('table', _p), ('pos_table', _p), ('pos_period', C.c_int32),
        ('const_row', _p), ('const_row2', _p), ('out_gamma', _p), ('out_beta', _p),
        ('eps', _f), ('y32', _p), ('y16', _p), ('rows', _l), ('a2', _p), ('a3', _p),
        ('y16_dtype', C.c_int32), ('ln2_gamma', _p), ('ln2_beta', _p), ('ln2_eps', _f), ('zero_rows', _l),
    ]


class GemmArgs(C.Structure):
    _fields_ = [('x', _p), ('ldx', _l), ('w', _p), ('in_dtype', _i), ('bias', _p), ('residual', _p), ('ldr', _l),
                ('y', _p), ('ldy', _l), ('y_dtype', _i), ('y16', _p), ('ldy16', _l),
                ('M', _i), ('N', _i), ('K', _i), ('epilogue', _i), ('n_groups', _i), ('group_row_end', _ip), ('tile', _i),
                ('ln_mode', _i), ('ln_vec_a', _p), ('ln_stats', _p), ('ln_chunks', _i), ('ln_eps', _f),
                ('stats_out', _p), ('stats_ld', _l)]


class AttnProblem(C.Structure):
    _fields_ = [('q', _p), ('ldq', _l), ('k', _p), ('ldk', _l), ('v', _p), ('ldv', _l), ('o', _p), ('ldo', _l),
                ('key_mask', _p), ('pair_dist', _p), ('bias_affine', _p), ('lse', _p),
                ('B', C.c_int32), ('Lq', C.c_int32), ('Lk', C.c_int32),
                ('drop_p', C.c_float), ('drop_site', C.c_uint32), ('drop_seed', _p)]


# name -> argtypes; every entry of include/vlnimagine.h must appear here (tests check the header against it)
PROTOTYPES = {
    'vi_version': [],
    'vi_launch_count': [],
    'vi_init': [_i],
    'vi_gemm16': [C.POINTER(GemmArgs), _p],
    'vi_gemm_f32': [_p, _l, _p, _p, _p, _l, _p, _l, _i, _i, _i, _i, _i, _ip, _p],
    'vi_attn_fwd_multi': [C.POINTER(AttnProblem), _i, _i, _i, _i, _p],
    'vi_add_ln': [_p, _p, _p, _p, _f, _p, _p, _i, _l, _i, _ip, _p],
    'vi_embed_compose': [C.POINTER(EmbedArgs), _p],
    'vi_ln_dot': [_p, _p, _p, _f, _p, _p, _p, _l, _i, _ip, _p],
    'vi_mul_bcast': [_p, _l, _p, _l, _p, _p, _i, _l, _i, _p],
    'vi_duet_fuse_logits': [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    'vi_mask_logits_navtype': [_p, _p, _p, _l, _p],
    'vi_gather_mean': [_p, _p, _p, _p, _p, _i, _i, _p],
    'vi_scatter_rows': [_p, _p, _p, _i, _p],
    'vi_cosine_loss': [_p, _p, _p, _p, _i, _p],
    'vi_infonce_loss': [_p, _p, _p, _p, _p, _f, _p, _p, _i, _i, _p],
    'vi_margin_loss': [_p, _p, _p, _p, _p, _f, _p, _p, _i, _i, _p],
    'vi_ce_rows': [_p, _l, _p, _i, _p, _l, _p],
    'vi_kl_rows': [_p, _l, _p, _l, _i, _p, _l, _p],
    'vi_ce_rows_bwd': [_p, _l, _p, _i, _p, _p, _p, _i, _l, _l, _p],
    'vi_kl_rows_bwd': [_p, _l, _p, _l, _i, _p, _p, _p, _i, _l, _l, _p],
    'vi_copy_rows': [_p, _l, _l, _p, _p, _i, _l, _l, _l, _i, _p],
    'vi_cast_h16': [_p, _p, _i, _l, _p],
    'vi_transpose': [_p, _l, _p, _l, _i, _i, _i, _i, _p],
    'vi_colsum': [_p, _l, _i, _p, _l, _i, _p, _l, _p],
    'vi_wgrad16_splits': [_i, _i, _i, _ip],
    'vi_wgrad16_workspace': [_i, _i, _i, _ip, _i],
    'vi_wgrad16': [_p, _l, _p, _l, _i, _i, _i, _i, _ip, _p, _p, _p, _l, _i, _i, _p],
    'vi_act_fwd': [_p, _p, _l, _i, _i, _p],
    'vi_act_bwd': [_p, _p, _p, _l, _i, _i, _p],
    'vi_add_ln_drop': [_p, _p, _p, _p, _f, _p, _p, _i, _l, _i, _ip, _f, _p, C.c_uint32, _p],
    'vi_add_ln_drop_bwd': [_p, _p, _p, _f, _p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _ip, _p, _l, _i, _f, _p, C.c_uint32, _p],
    'vi_feat_wgrad': [_p, _p, _i, _p, _p, _l, _p, _l, _p],
    'vi_scatter_add_rows': [_p, _p, _i, _p, _l, _p],
    'vi_rowdot_bwd': [_p, _p, _p, _p, _p, _p, _l, _i, _ip, _p, _l, _p],
    'vi_attn_bwd': [_p, _l, _p, _l, _p, _l, _p, _l, _p, _l, _p, _l, _p, _l, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, C.c_uint32, _p, _p],
    'vi_dropout': [_p, _p, _l, _f, _p, C.c_uint32, _i, _p],
    'vi_duet_fuse_logits_bwd': [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    'vi_mul_bcast_bwd_s': [_p, _p, _p, _l, _i, _p],
    'vi_cosine_loss_bwd': [_p, _p, _p, _p, _p, _i, _p],
    'vi_infonce_loss_bwd': [_p, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p, _i, _i, _p],
    'vi_margin_loss_bwd': [_p, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p, _i, _i, _p],
    'vi_graph_init': [_p, _p, _p, _p, _i, _i, _p],
    'vi_graph_update': [_p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _i, _p, _p],
    'vi_graph_embed_step': [_p, _p, _i, _i, _i, _p, _p, _i, _p, _p, _p, _i, _p, _i, _p, _p, _p],
    'vi_graph_features': [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _i, _p, _p, _p, _i, _p, _i, _p, _p],
}
# entry points that return a value rather than a VI_OK / VI_ERR_* status (ops.lib passes their result through unchecked)
QUERIES = {'vi_version', 'vi_wgrad16_splits', 'vi_wgrad16_workspace', 'vi_launch_count', 'vi_last_error'}
for _name, _args in PROTOTYPES.items():
    _fn = getattr(lib, _name)            # AttributeError here = header/library mismatch: fail loudly
    _fn.argtypes = _args
    _fn.restype = _i
lib.vi_wgrad16_workspace.restype = C.c_int64
lib.vi_launch_count.restype = C.c_int64
lib.vi_last_error.argtypes = []
lib.vi_last_error.restype = C.c_char_p


class VlnImagineError(RuntimeError):
    pass


def failure(rc: int, what: str = '') -> VlnImagineError:
    return VlnImagineError('%s failed (%d): %s' % (what or 'libvlnimagine call', rc, lib.vi_last_error().decode()))


def check(rc: int, what: str = ''):
    if rc != VI_OK:
        raise failure(rc, what)


def int_array(values):
    if values is None:
        return None
    return (C.c_int32 * len(values))(*values)
