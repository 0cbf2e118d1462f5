"""ctypes binding of the C-ABI library ``libnnr_b200.so`` (declared in ``include/nnr_b200.h``).

The library is built in-tree by ``nnr_b200/csrc/build.sh`` (``__graft_entry__.build()``).  There is
no fallback: if the shared object is missing the import fails, and every op raises on non-CUDA
tensors.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# NNR_B200_LIB: another build of the same library (the -DNNR_TC_PROF / -DNNR_LSTM_PROF instrumented ones of scripts/*_prof.py)
LIB_PATH = os.environ.get('NNR_B200_LIB') or os.path.join(_HERE, '_lib', 'libnnr_b200.so')

if not os.path.isfile(LIB_PATH):
    raise ImportError('nnr_b200: CUDA library not built (%s missing). Run nnr_b200/csrc/build.sh or '
                      '__graft_entry__.build(); there is no CPU fallback.' % LIB_PATH)

lib = C.CDLL(LIB_PATH)

vp, i32, i64, u64, f32, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_size_t


class GemmArgs(C.Structure):
    _fields_ = [('A', vp), ('lda', i64), ('transA', i32),
                ('B', vp), ('ldb', i64), ('transB', i32),
                ('C', vp), ('ldc', i64),
                ('M', i32), ('N', i32), ('K', i32),
                ('m_dev', vp), ('k_dev', vp),
                ('epilogue', i32), ('accumulate', i32),
                ('bias', vp), ('aux', vp), ('ldaux', i64),
                ('aux_out', vp), ('ldaux_out', i64),
                ('rowbias', vp), ('ldrowbias', i64), ('rowmap', vp),
                ('p_drop', f32), ('seed', u64),
                ('algo', i32),
                ('workspace', vp), ('workspace_bytes', sz),
                ('A_planes', vp), ('a_planes_pitch', i64), ('a_planes_rows', i64),
                ('B_planes', vp), ('b_planes_pitch', i64), ('b_planes_rows', i64),
                ('C_planes', vp), ('c_planes_pitch', i64), ('c_planes_rows', i64)]


class PoolArgs(C.Structure):
    _fields_ = [('X', vp), ('ldx', i64), ('D', i32),
                ('seg_off', vp), ('S', i32), ('fixed_len', i32), ('max_len', i32),
                ('mode', i32),
                ('U', vp), ('ldu', i64), ('A', i32), ('w2', vp),
                ('qvec', vp), ('ldq', i64), ('scale', f32),
                ('mask', vp),
                ('pooled', vp), ('ldp', i64),
                ('alpha', vp),
                ('dpooled', vp), ('lddp', i64),
                ('dX', vp), ('lddx', i64), ('accumulate_dx', i32),
                ('dU', vp), ('lddu', i64),
                ('dw2_partial', vp),
                ('dqvec', vp), ('lddq', i64),
                ('seg_order', vp)]


class SplitDesc(C.Structure):
    _fields_ = [('src', vp), ('ld', i64), ('rows', i32), ('cols', i32), ('planes', vp), ('pitch', i64)]


# name -> (restype, argtypes); must list every symbol include/nnr_b200.h declares
SIGNATURES = {
    'nnr_last_error': (C.c_char_p, []),
    'nnr_abi_version': (C.c_int, []),
    'nnr_launch_count': (u64, []),
    'nnr_profile_enable': (C.c_int, [C.c_int]),
    'nnr_profile_read': (C.c_int, [C.POINTER(C.c_double), C.c_int]),
    'nnr_seq_prepare': (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp]),
    'nnr_embed_gather_fwd': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, f32, u64, vp]),
    'nnr_embed_gather_planes_fwd': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32, u64, C.c_int, vp, sz, vp]),
    'nnr_embed_gather_bwd_workspace_bytes': (sz, [C.c_int, C.c_int]),
    'nnr_embed_gather_bwd': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, f32, u64, vp, C.c_int, vp, sz, vp]),
    'nnr_gemm_workspace_bytes': (sz, [C.POINTER(GemmArgs)]),
    'nnr_gemm': (C.c_int, [C.POINTER(GemmArgs), vp]),
    'nnr_tc_split_pitch': (i64, [C.c_int, C.c_int]),
    'nnr_tc_split_bytes': (sz, [C.c_int, C.c_int, C.c_int]),
    'nnr_tc_split': (C.c_int, [vp, i64, C.c_int, C.c_int, vp, C.c_int, vp, sz, vp]),
    'nnr_tc_split_colsum_workspace_bytes': (sz, [C.c_int, C.c_int, C.c_int]),
    'nnr_tc_split_colsum': (C.c_int, [vp, i64, C.c_int, C.c_int, vp, C.c_int, vp, sz, vp, C.c_int, vp, sz, vp]),
    'nnr_relu_bwd_split_colsum': (C.c_int, [vp, vp, i64, C.c_int, C.c_int, f32, u64, vp, C.c_int, vp, sz, vp, C.c_int, vp, sz, vp]),
    'nnr_length_sort_desc': (C.c_int, [vp, C.c_int, C.c_int, vp, vp]),
    'nnr_tc_split_many': (C.c_int, [vp, C.c_int, C.c_int, vp]),
    'nnr_gemm_default_algo': (C.c_int, []),
    'nnr_colsum_workspace_bytes': (sz, [C.c_int, C.c_int]),
    'nnr_colsum': (C.c_int, [vp, i64, C.c_int, C.c_int, vp, vp, C.c_int, vp, sz, vp]),
    'nnr_segment_colsum': (C.c_int, [vp, i64, vp, C.c_int, C.c_int, vp, i64, vp]),
    'nnr_lstm_fwd': (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    'nnr_lstm_bwd': (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    'nnr_lstm_bwd_planes_supported': (C.c_int, [C.c_int, C.c_int]),
    'nnr_lstm_fwd_planes_supported': (C.c_int, [C.c_int, C.c_int]),
    'nnr_lstm_fwd_planes': (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, vp, sz, vp]),
    'nnr_lstm_bwd_planes_workspace_bytes': (sz, [C.c_int, C.c_int]),
    'nnr_lstm_bwd_planes': (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_int, vp, sz, vp,
                                      vp, sz, vp]),
    'nnr_lstm_shift_h_planes': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, sz, vp]),
    'nnr_lstm_shift_h': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp]),
    'nnr_gate_bwd_planes': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, sz, vp, vp, i64, vp]),
    'nnr_gate_bwd_pre': (C.c_int, [vp, vp, vp, i64, vp, C.c_int, vp, vp, vp]),
    'nnr_attn_pool_fwd': (C.c_int, [C.POINTER(PoolArgs), vp]),
    'nnr_attn_pool_bwd': (C.c_int, [C.POINTER(PoolArgs), vp]),
    'nnr_news_fuse_fwd': (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, f32, u64, vp, vp]),
    'nnr_news_fuse_bwd': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32, u64, vp, vp, vp, vp, C.c_int, vp]),
    'nnr_news_fuse_tables_bwd': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32, u64, vp, vp, C.c_int, vp]),
    'nnr_sue_graph_build': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    'nnr_sue_graph_build_ex': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    'nnr_ln_relu_res_fwd': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, f32, f32, u64, vp, vp, vp, vp, vp]),
    'nnr_ln_relu_res_bwd_workspace_bytes': (sz, [C.c_int, C.c_int]),
    'nnr_ln_relu_res_bwd': (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, f32, u64, vp, vp, vp, vp, vp, sz, vp]),
    'nnr_graph_to_csr': (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    'nnr_gcn_aggregate': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp]),
    'nnr_gcn_aggregate_add': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    'nnr_cluster_intra_fwd': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32, vp, vp, vp]),
    'nnr_cluster_intra_bwd': (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32, vp, vp, vp, vp, C.c_int, vp]),
    'nnr_cluster_tail_scores': (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, f32, vp, i64, vp]),
    'nnr_cluster_tail_scores_packed': (C.c_int, [vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int,
                                                 C.c_int, C.c_int, C.c_int, f32, vp, i64, vp]),
    'nnr_cluster_tail_explain_packed': (C.c_int, [vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int,
                                                  C.c_int, C.c_int, C.c_int, f32, vp, i64, vp, vp, vp, vp]),
    'nnr_rowdot_fwd': (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp]),
    'nnr_rowdot_bwd': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp, C.c_int, vp]),
    'nnr_topk_merge': (C.c_int, [vp, i64, C.c_int, C.c_int, i64, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    'nnr_topk_merge_capped': (C.c_int, [vp, i64, C.c_int, C.c_int, i64, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int,
                                        C.c_int, vp, vp, vp, vp]),
    'nnr_topk_merge_lists': (C.c_int, [vp, i64, C.c_int, C.c_int, vp, i64, C.c_int, C.c_int, vp, vp, vp]),
    'nnr_topk_merge_lists_capped': (C.c_int, [vp, i64, C.c_int, C.c_int, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int,
                                              vp, vp, vp, vp]),
    'nnr_dropout': (C.c_int, [vp, i64, f32, u64, vp, vp]),
    'nnr_flat_clip_adam_workspace_bytes': (sz, [i64]),
    'nnr_flat_clip_adam': (C.c_int, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, i32, vp, vp, sz, vp]),
    'nnr_flat_clip_adam_dev': (C.c_int, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, vp, vp, vp, sz, vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here == header/library mismatch
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc, what):
    if rc != 0:
        msg = lib.nnr_last_error()
        raise RuntimeError('%s failed (rc=%d): %s' % (what, rc, msg.decode() if msg else ''))


def launch_count():
    return int(lib.nnr_launch_count())
