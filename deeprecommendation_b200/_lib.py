"""ctypes binding of libb200rec.so (include/b200rec.h).  There is no fallback: if the library is missing or no
CUDA device is present, every op raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('B200REC_LIB') or os.path.join(_HERE, 'libb200rec.so')     # (B200REC_LIB: an experimental build of the same ABI, A/B measurements)

OK, ERR_CUDA, ERR_BAD_ARG, ERR_UNSUPPORTED, ERR_WORKSPACE = 0, 1, 2, 3, 4
F32, BF16 = 0, 1
ATT_NET, ATT_DOT = 0, 1
TC_TF32X3, TC_BF16, TC_BF16X3 = 0, 1, 2
ABI_VERSION = 209          # B200REC_VERSION of include/b200rec.h these bindings were written against (checked when the library is loaded)
AP_BF16, AP_BF16X2 = 0, 1
MLP_MAX_LAYERS = 8
PEER_MAX, PEER_CHANNELS, PEER_HANDLE_BYTES = 16, 16, 64

c_i64, c_int, c_sz, c_vp, c_f = C.c_int64, C.c_int, C.c_size_t, C.c_void_p, C.c_float


class MlpDesc(C.Structure):
    _fields_ = [('W', c_vp * MLP_MAX_LAYERS), ('b', c_vp * MLP_MAX_LAYERS), ('out_dim', c_int * MLP_MAX_LAYERS),
                ('n_layers', c_int)]


class AttentionDesc(C.Structure):
    _fields_ = [('Pc', c_vp), ('Pr', c_vp), ('Q', c_vp), ('table_dtype', c_int), ('mode', c_int), ('a2', c_vp), ('a20', c_vp),
                ('bU', c_vp), ('user_matrix', c_vp), ('ld_user_matrix', c_i64), ('row_ptr', c_vp), ('col', c_vp), ('val', c_vp),
                ('B', c_i64), ('I', c_i64), ('H', c_int), ('U', c_int), ('out', c_vp), ('ldo', c_i64), ('att_weights', c_vp),
                ('train_cand_emb', c_vp), ('train_rated_emb', c_vp), ('E', c_int), ('atol', c_f), ('rtol', c_f),
                ('drop_zero_scores', c_int), ('score_scale', c_f), ('ld_pr', c_i64), ('ld_q', c_i64), ('workspace', c_vp), ('workspace_bytes', c_sz),
                ('max_row_nnz', c_i64), ('nnz', c_i64), ('ld_pc', c_i64), ('dropout_p', c_f), ('dropout_seed', C.c_uint64), ('dropout_seed_dev', c_vp)]


class AttentionBwdDesc(C.Structure):
    _fields_ = [('Pc', c_vp), ('Pr', c_vp), ('Q', c_vp), ('mode', c_int), ('a2', c_vp), ('bU', c_vp), ('user_matrix', c_vp), ('ld_user_matrix', c_i64),
                ('att_weights', c_vp), ('out', c_vp), ('ldo', c_i64), ('grad_out', c_vp), ('ld_grad_out', c_i64), ('B', c_i64), ('I', c_i64),
                ('H', c_int), ('U', c_int), ('score_scale', c_f), ('ld_pc', c_i64), ('ld_pr', c_i64), ('ld_q', c_i64),
                ('dPc', c_vp), ('dPr', c_vp), ('dQ', c_vp), ('da2_rows', c_vp), ('da20_rows', c_vp), ('n_slices', c_int), ('dropout_p', c_f),
                ('dropout_seed', C.c_uint64), ('dropout_seed_dev', c_vp)]


class LinearProblem(C.Structure):
    _fields_ = [('X', c_vp), ('M', c_i64), ('ldx', c_i64), ('W', c_vp), ('N', c_i64), ('ldw', c_i64), ('packed_w', c_vp), ('bias', c_vp),
                ('row_scale', c_vp), ('relu', c_int), ('Y', c_vp), ('ldy', c_i64), ('y_dtype', c_int)]


class SpmmDesc(C.Structure):
    _fields_ = [('chunk_row', c_vp), ('chunk_start', c_vp), ('chunk_slot', c_vp), ('n_chunks', c_int), ('chunk_size', c_int),
                ('row_ptr', c_vp), ('col', c_vp), ('w', c_vp), ('perm', c_vp), ('skip_bits', c_vp), ('t', c_vp), ('t_dtype', c_int),
                ('ld_t', c_i64), ('d', c_int), ('dinv', c_vp), ('partials', c_vp), ('x_next', c_vp), ('ld_x', c_i64),
                ('acc_in', c_vp), ('acc_out', c_vp), ('ld_acc', c_i64), ('acc_scale', c_f), ('multi_row', c_vp),
                ('multi_first_slot', c_vp), ('multi_n_slots', c_vp), ('n_multi', c_int), ('att_src', c_vp), ('partials_ml', c_vp),
                ('push_dst', c_vp * PEER_MAX), ('push_parts', c_int), ('push_rows_per_part', c_int), ('push_offset', c_i64), ('push_ld', c_i64),
                ('push_stats_offset', c_i64)]


class SpmmStreamDesc(C.Structure):
    _fields_ = [('colf', c_vp), ('wd', c_vp), ('nnz', c_i64), ('seg', c_int), ('n_segs', c_int), ('seg_first_j', c_vp), ('seg_head_slot', c_vp),
                ('seg_tail_slot', c_vp), ('rows_ne', c_vp), ('n_ne', c_int), ('rows_empty', c_vp), ('n_empty', c_int), ('t', c_vp), ('t_dtype', c_int),
                ('ld_t', c_i64), ('d', c_int), ('partials', c_vp), ('multi_row', c_vp), ('multi_first_slot', c_vp), ('multi_n_slots', c_vp),
                ('n_multi', c_int), ('x_next', c_vp), ('ld_x', c_i64), ('acc_in', c_vp), ('acc_out', c_vp), ('ld_acc', c_i64), ('acc_scale', c_f),
                ('push_dst', c_vp * PEER_MAX), ('push_parts', c_int), ('push_rows_per_part', c_int), ('push_offset', c_i64), ('push_ld', c_i64)]


# name -> (restype, argtypes); this table is also what tests/test_abi.py checks against include/b200rec.h
SIGNATURES = {
    'b200rec_last_error': (C.c_char_p, []),
    'b200rec_version': (c_int, []),
    'b200rec_sm_count': (c_int, []),
    'b200rec_launch_count': (c_i64, []),
    'b200rec_linear_workspace': (c_sz, [c_i64, c_i64, c_i64]),
    'b200rec_linear': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_vp, c_sz, c_vp]),
    'b200rec_linear_tc_splitk_workspace': (c_sz, [c_i64, c_i64, c_i64, c_int]),
    'b200rec_linear_tc_splitk': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_linear_tc': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_i64, c_vp]),
    'b200rec_linear_tc_wide_workspace': (c_sz, [c_i64, c_i64, c_i64, c_int]),
    'b200rec_linear_tc_wide': (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    'b200rec_linear_shortk': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_vp]),
    'b200rec_linear_shortk_push': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_int, C.POINTER(c_vp), c_int, c_i64, c_i64, c_int, c_vp]),
    'b200rec_linear_sparse': (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_i64, c_int, c_vp]),
    'b200rec_dense_nnz_count': (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp]),
    'b200rec_dense_nnz_fill': (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    'b200rec_linear_tc_batch': (c_int, [C.POINTER(LinearProblem), c_int, c_i64, c_int, c_vp]),
    'b200rec_linear_tc_splitk_batch_workspace': (c_sz, [C.POINTER(LinearProblem), c_int, c_i64, c_int]),
    'b200rec_linear_tc_splitk_batch': (c_int, [C.POINTER(LinearProblem), c_int, c_i64, c_int, c_vp, c_sz, c_vp]),
    'b200rec_packed_weight_bytes': (c_sz, [c_i64, c_i64, c_int]),
    'b200rec_pack_weights_tc': (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_sz, c_vp]),
    'b200rec_mlp_tower': (c_int, [c_vp, c_i64, c_vp, c_int, c_vp, c_i64, c_vp, c_int, c_i64, C.POINTER(MlpDesc), c_vp, c_i64, c_vp]),
    'b200rec_rowdot': (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_int, c_i64, c_vp, c_vp]),
    'b200rec_allpairs_packed_bytes': (c_sz, [c_int, c_int]),
    'b200rec_allpairs_pack': (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_vp, c_sz, c_vp]),
    'b200rec_allpairs_splits': (c_int, [c_i64, c_i64, c_int]),
    'b200rec_allpairs_workspace': (c_sz, [c_i64, c_int, c_int]),
    'b200rec_allpairs_topk': (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_allpairs_relu_dot_splits': (c_int, [c_i64, c_i64]),
    'b200rec_allpairs_relu_dot_topk': (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_f, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_allpairs_dot_topk': (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_topk_rows': (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp]),
    'b200rec_attention_pool_workspace': (c_sz, [c_i64, c_i64, c_int, c_int]),
    'b200rec_attention_pool_workspace_csr': (c_sz, [c_i64, c_i64, c_int, c_i64, c_i64]),
    'b200rec_attention_pool': (c_int, [C.POINTER(AttentionDesc), c_vp]),
    'b200rec_attention_pool_dropout': (c_int, [C.POINTER(AttentionDesc), c_vp]),
    'b200rec_attention_pool_set_path': (c_int, [c_int]),
    'b200rec_attention_pool_backward': (c_int, [C.POINTER(AttentionBwdDesc), c_vp]),
    'b200rec_attention_recommend_workspace': (c_sz, [c_i64, c_i64, c_int]),
    'b200rec_attention_recommend': (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_i64, c_vp, c_vp, c_vp,
                                            c_vp, c_i64, c_vp, c_i64, c_vp]),
    'b200rec_attention_recommend_bf16': (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_i64, c_vp, c_vp,
                                                 c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    'b200rec_attention_explain_workspace': (c_sz, [c_i64, c_int]),
    'b200rec_attention_explain_count': (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_int,
                                                C.c_double, C.c_double, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_attention_explain_fill': (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_int,
                                               c_vp, c_vp, c_sz, c_vp, c_vp, c_vp]),
    'b200rec_spmm': (c_int, [C.POINTER(SpmmDesc), c_vp]),
    'b200rec_spmm_stream': (c_int, [C.POINTER(SpmmStreamDesc), c_vp]),
    'b200rec_scan_workspace': (c_sz, [c_i64]),
    'b200rec_exclusive_scan_i32': (c_int, [c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_sort_pairs_workspace': (c_sz, [c_i64]),
    'b200rec_sort_pairs_i32': (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_sz, c_vp]),
    'b200rec_id_rank_table': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_id_lookup': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    'b200rec_group_stats': (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    'b200rec_edge_attrs': (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rec_edge_scatter': (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]),
    'b200rec_csr_workspace': (c_sz, [c_i64, c_i64]),
    'b200rec_csr_build': (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_dinv': (c_int, [c_vp, c_i64, c_vp, c_vp]),
    'b200rec_spmm_plan_workspace': (c_sz, [c_i64]),
    'b200rec_spmm_plan_count': (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_spmm_plan_fill': (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rec_pairhash_build': (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    'b200rec_pairhash_lookup': (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    'b200rec_mask_targets': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rec_collate_workspace': (c_sz, [c_i64, c_i64]),
    'b200rec_collate_interacted': (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    'b200rec_sample_negatives': (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, C.c_double, C.c_uint64, C.c_uint64, c_vp, c_vp, c_vp, c_vp]),
    'b200rec_peer_alloc': (c_int, [c_sz, C.POINTER(c_vp), C.c_char_p]),
    'b200rec_peer_open': (c_int, [C.c_char_p, C.POINTER(c_vp)]),
    'b200rec_peer_close': (c_int, [c_vp]),
    'b200rec_peer_free': (c_int, [c_vp]),
    'b200rec_peer_signal': (c_int, [C.POINTER(c_vp), c_int, c_int, c_int, c_vp, c_vp]),
    'b200rec_peer_wait': (c_int, [c_vp, c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    'b200rec_peer_reduce': (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_vp, c_vp, c_i64, c_f, c_vp]),
    'b200rec_peer_reduce_softmax': (c_int, [c_vp, c_vp, c_int, c_i64, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_vp, c_vp, c_i64, c_f, c_vp]),
    'b200rec_peer_push_floats': (c_int, [c_vp, c_i64, C.POINTER(c_vp), c_int, c_i64, c_vp]),
    'b200rec_peer_push_rows': (c_int, [c_vp, c_i64, c_i64, c_int, C.POINTER(c_vp), c_int, c_i64, c_i64, c_vp]),
    'b200rec_device_timestamp': (c_int, [c_vp, c_vp]),
    'b200rec_peer_scale_rows': (c_int, [c_vp, c_i64, c_i64, c_int, c_vp, c_i64, c_vp, c_f, c_vp, c_i64, c_vp, c_i64, c_vp]),
    'b200rec_peer_rows_to_owned': (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_f, c_vp, c_i64, c_vp]),
    'b200rec_peer_mask_targets': (c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rec_peer_gather_rows': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_f, C.POINTER(c_vp), c_int, c_i64, c_i64, c_vp]),
}

_lib = None


class B200RecError(RuntimeError):
    pass


def lib():
    """Loads libb200rec.so (once).  Raises — never falls back — when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f'{LIB_PATH} not found: build the CUDA library first (python -m deeprecommendation_b200.csrc.build, or '
                f'__graft_entry__.build()).  deeprecommendation_b200 has no CPU / PyTorch fallback.')
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)          # AttributeError here = header / library out of sync
            fn.restype, fn.argtypes = res, args
        if h.b200rec_version() != ABI_VERSION:      # a stale build of an older header: struct layouts / signatures would not match
            raise ImportError(f'{LIB_PATH} reports ABI version {h.b200rec_version()}, these bindings need {ABI_VERSION}: rebuild it '
                              f'(python -m deeprecommendation_b200.csrc.build --force)')
        _lib = h
    return _lib


def check(rc: int, what: str = ''):
    if rc != OK:
        msg = lib().b200rec_last_error().decode(errors='replace')
        kind = {ERR_CUDA: 'CUDA', ERR_BAD_ARG: 'bad argument', ERR_UNSUPPORTED: 'unsupported', ERR_WORKSPACE: 'workspace'}.get(rc, str(rc))
        if rc == ERR_UNSUPPORTED:
            raise NotImplementedError(f'b200rec {what}: {msg}')
        if rc == ERR_BAD_ARG:
            raise ValueError(f'b200rec {what}: {msg}')
        raise B200RecError(f'b200rec {what} failed ({kind}): {msg}')
