"""ctypes binding of ``librlzero_b200.so`` (the C ABI in ``include/rlzero_b200.h``).

There is deliberately NO fallback: if the CUDA library is missing, cannot be loaded, or
disagrees with this file about the ABI, importing the product path raises.
"""
import ctypes as C
import os

import torch  # noqa: F401  -- loads libcudart.so.12 into the process before our library

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'librlzero_b200.so')

ABI_VERSION = 14
META_STRIDE = 12
(META_PLAYER, META_LAST_MOVE, META_STONES, META_STATUS, META_WINNER, META_PLY, META_FAULT,
 META_EPISODE, META_KO, META_PASSES) = range(10)
GO_HIST = 14
ACTIVE, ENDED_WIN, ENDED_TIE, IDLE = range(4)
FAULT_ILLEGAL_MOVE, FAULT_POOL_OVERFLOW, FAULT_DEPTH_OVERFLOW, FAULT_LN_TABLE = 1, 2, 4, 8
FAULT_NO_CHILDREN, FAULT_CARRY_DROPPED, FAULT_TRAJ_OVERFLOW = 16, 32, 64
RULE_UCT, RULE_PUCT = 0, 1
FLAVOUR_ALPHAZERO, FLAVOUR_DEEPMIND = 0, 1
RETURNS_REFERENCE, RETURNS_ZERO_SUM = 0, 1
EVAL_ZERO, EVAL_KAT, EVAL_HASH = 0, 1, 2
CHILD_TERMINAL, CHILD_OVERFLOW, CHILD_PENDING = -1, -2, -3
MAX_BOARD = 19

_vp = C.c_void_p


GAME_GOMOKU, GAME_CONNECT4, GAME_GO = 0, 1, 2


class GameDesc(C.Structure):
    """rz_game_desc: GameDesc(H, k, A, AS[, W, game_type, komi, max_moves, row_stride]); W = 0 means a square
    board, row_stride = 0 the automatic padded layout of the network kernels (see row_stride())."""
    _fields_ = [('board_size', C.c_int32), ('n_in_row', C.c_int32), ('n_actions', C.c_int32),
                ('action_stride', C.c_int32), ('width', C.c_int32), ('game_type', C.c_int32),
                ('komi', C.c_float), ('max_moves', C.c_int32), ('row_stride', C.c_int32)]


class TreeDesc(C.Structure):
    _fields_ = [('game', GameDesc), ('n_trees', C.c_int32), ('max_nodes', C.c_int32),
                ('max_depth', C.c_int32), ('rule', C.c_int32), ('ln_table_len', C.c_int32),
                ('store_priors', C.c_int32), ('c_puct', C.c_double), ('global_offset', C.c_int64),
                ('edge_N', _vp), ('edge_W', _vp), ('edge_P', _vp), ('edge_child', _vp),
                ('node_parent', _vp), ('node_paction', _vp),
                ('n_nodes', _vp), ('root_N', _vp), ('root_W', _vp),
                ('root_rows', _vp), ('root_meta', _vp),
                ('path_node', _vp), ('path_action', _vp), ('depth', _vp),
                ('leaf_rows', _vp), ('leaf_meta', _vp), ('ln_table', _vp),
                ('root_hist', _vp), ('leaf_hist', _vp),
                ('flavour', C.c_int32), ('solve', C.c_int32), ('returns_mode', C.c_int32),
                ('noise_root_only', C.c_int32), ('edge_O', _vp), ('root_O', _vp),
                ('leaves_per_tree', C.c_int32), ('target_N', _vp), ('vl_saved_W', _vp),
                ('virtual_loss', C.c_double),
                ('edge_P64', _vp), ('seed_dev', _vp), ('edge_R', _vp), ('shuffle_mode', C.c_int32),
                ('reserved0', C.c_int32)]


class TrajDesc(C.Structure):
    _fields_ = [('max_plies', C.c_int32), ('ring_capacity', C.c_int32),
                ('stage_rows', _vp), ('stage_info', _vp), ('stage_pi', _vp),
                ('ring_rows', _vp), ('ring_info', _vp), ('ring_pi', _vp),
                ('ring_cursor', _vp), ('games_done', _vp), ('plies_done', _vp)]


class MzDesc(C.Structure):
    """rz_mz_desc: MuZero latent-space trees."""
    _fields_ = [('n_trees', C.c_int32), ('n_actions', C.c_int32), ('action_stride', C.c_int32),
                ('max_nodes', C.c_int32), ('max_depth', C.c_int32), ('pbc_table_len', C.c_int32),
                ('discount', C.c_double), ('known_min', C.c_double), ('known_max', C.c_double),
                ('global_offset', C.c_int64),
                ('edge_N', _vp), ('edge_W', _vp), ('edge_P', _vp), ('edge_child', _vp),
                ('n_nodes', _vp), ('root_N', _vp), ('root_W', _vp), ('mm_min', _vp), ('mm_max', _vp),
                ('path_node', _vp), ('path_action', _vp), ('depth', _vp), ('leaf_parent', _vp),
                ('leaf_action', _vp), ('fault', _vp), ('pbc_table', _vp)]


class HeadsDesc(C.Structure):
    _fields_ = [('board_size', C.c_int32), ('action_stride', C.c_int32), ('width', C.c_int32),
                ('n_actions', C.c_int32), ('row_stride', C.c_int32), ('w1x1', _vp), ('b1x1', _vp), ('wp', _vp), ('bp', _vp),
                ('wv1', _vp), ('bv1', _vp), ('wv2', _vp), ('bv2', _vp), ('wtc_hi', _vp), ('wtc_lo', _vp)]


# name -> (restype, argtypes); every symbol include/rlzero_b200.h declares
_GD, _TD, _TJ = C.POINTER(GameDesc), C.POINTER(TreeDesc), C.POINTER(TrajDesc)
SIGNATURES = {
    'rz_abi_version': (C.c_int, []),
    'rz_last_error': (C.c_char_p, []),
    'rz_sizeof_tree_desc': (C.c_int, []),
    'rz_sizeof_traj_desc': (C.c_int, []),
    'rz_gomoku_reset': (C.c_int, [_GD, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_gomoku_step': (C.c_int, [_GD, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_gomoku_legal_mask': (C.c_int, [_GD, _vp, _vp, C.c_int, _vp]),
    'rz_gomoku_winner': (C.c_int, [_GD, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_gomoku_encode_f32': (C.c_int, [_GD, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_gomoku_encode_nhwc_f32': (C.c_int, [_GD, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_go_reset': (C.c_int, [_GD, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_go_step': (C.c_int, [_GD, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_go_legal_mask': (C.c_int, [_GD, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_go_score': (C.c_int, [_GD, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_go_encode_f32': (C.c_int, [_GD, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_tree_reset': (C.c_int, [_TD, _vp, _vp]),
    'rz_tree_select': (C.c_int, [_TD, _vp]),
    'rz_tree_expand_backup': (C.c_int, [_TD, _vp, C.c_int, _vp, _vp, C.c_float, C.c_float,
                                        C.c_ulonglong, _vp]),
    'rz_tree_expand_backup_select': (C.c_int, [_TD, _vp, C.c_int, _vp, _vp, C.c_float, C.c_float,
                                               C.c_ulonglong, _vp]),
    'rz_tree_expand_backup_ex': (C.c_int, [_TD, _vp, C.c_int, _vp, _vp, C.c_float, C.c_float,
                                           C.c_ulonglong, _vp, _vp, _vp]),
    'rz_tree_expand_backup_dm': (C.c_int, [_TD, _vp, C.c_int, _vp, _vp, C.c_float, C.c_float,
                                           C.c_ulonglong, _vp]),
    'rz_tree_best_child': (C.c_int, [_TD, _vp, _vp, _vp]),
    'rz_tree_root_policy': (C.c_int, [_TD, C.c_double, _vp, _vp, _vp, _vp, C.c_ulonglong, _vp]),
    'rz_tree_advance': (C.c_int, [_TD, _vp, C.c_int, C.c_int, _TJ, _vp, C.c_int, _vp]),
    'rz_match_commit': (C.c_int, [_TD, _TD, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_eval_closed_form': (C.c_int, [_TD, C.c_int, _vp, _vp, _vp]),
    'rz_augment_equi': (C.c_int, [_GD, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_gather_rows': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_go_records_pack': (C.c_int, [_GD, _vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_go_records_expand': (C.c_int, [_GD, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'rz_learn_sgemm': (C.c_int, [C.c_int, C.c_int, C.c_int, _vp, C.c_longlong, C.c_longlong, _vp, C.c_longlong,
                                 C.c_longlong, _vp, C.c_longlong, C.c_float, C.c_int, _vp]),
    'rz_learn_colsum': (C.c_int, [_vp, C.c_longlong, C.c_int, C.c_longlong, _vp, C.c_float, _vp, C.c_int, _vp]),
    'rz_learn_pack_conv': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_learn_relu_bwd': (C.c_int, [_vp, _vp, C.c_longlong, _vp]),
    'rz_learn_nchw_to_nhwc': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_conv_wgrad': (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_head_feat_fwd': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_learn_logsoftmax': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_value_fwd': (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_learn_loss_bwd': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int,
                                    C.c_int, C.c_int, _vp]),
    'rz_learn_head_feat_bwd': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_int, _vp]),
    'rz_learn_adam': (C.c_int, [_vp, _vp, _vp, _vp, C.c_longlong, C.c_float, C.c_float, C.c_float, C.c_float,
                                C.c_float, C.c_int, _vp]),
    'rz_learn_conv_wgrad_tc': (C.c_int, [_vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_int, _vp]),
    'rz_learn_pack_conv_tc': (C.c_int, [_vp, _vp, _vp, _vp]),
    'rz_learn_pack_stem_tc': (C.c_int, [_vp, _vp, _vp]),
    'rz_net_pack_conv_bn_tc': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_float, _vp, _vp, _vp]),
    'rz_learn_bn_forward': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp, C.c_int, C.c_int,
                                      C.c_int, _vp]),
    'rz_learn_bn_backward': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_relu_bwd_bf16': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp]),
    'rz_learn_planes_to_tile': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_tile_colsum': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp]),
    'rz_learn_nhwc_to_tile_hilo': (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_nhwc_to_tile_hilo_slice': (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_tile_f32_to_nhwc': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_tile_grad_mask_split': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp]),
    'rz_learn_tile_to_nhwc': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_nhwc_to_tile': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_conv_wgrad_tc_ex': (C.c_int, [_vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_pack_stem_tc_ex': (C.c_int, [_vp, C.c_int, _vp, _vp]),
    'rz_learn_bn_forward_ex': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp, C.c_int,
                                         C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_bn_backward_ex': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                          _vp]),
    'rz_learn_planes_to_tile_ex': (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_tile_colsum_ex': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_learn_relu_bwd_bf16_ex': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    'rz_learn_tile_to_nhwc_ex': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_learn_nhwc_to_tile_ex': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_eval_rollout': (C.c_int, [_TD, C.c_int, C.c_ulonglong, C.c_int, _vp, _vp, _vp]),
    'rz_eval_rollout_dm': (C.c_int, [_TD, C.c_int, C.c_ulonglong, C.c_int, _vp, _vp, _vp]),
    'rz_sizeof_mz_desc': (C.c_int, []),
    'rz_mz_root': (C.c_int, [C.POINTER(MzDesc), _vp, _vp, C.c_float, C.c_float, C.c_ulonglong, C.c_uint, _vp, _vp]),
    'rz_mz_select': (C.c_int, [C.POINTER(MzDesc), _vp]),
    'rz_mz_expand_backup': (C.c_int, [C.POINTER(MzDesc), _vp, _vp, _vp]),
    'rz_mz_gather': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, _vp]),
    'rz_net_conv3x3_tc2': (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int, _vp]),
    'rz_debug_set_probe': (C.c_int, [_vp]),
    'rz_net_trunk_small_ex': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_int,
                                         C.c_int, C.c_int, _vp, _vp, _vp, _vp]),
    'rz_net_trunk_small': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_uint, C.c_uint, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp,
                                      _vp]),
    'rz_net_trunk_tc2': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_uint, C.c_uint, _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                   _vp, _vp, _vp, C.c_int, _vp]),
    'rz_net_conv3x3_tc2_head_ex': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             _vp, _vp, _vp, C.c_int, _vp]),
    'rz_net_conv3x3_tc3': (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, _vp]),
    'rz_net_conv3x3_tc3_head': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp,
                                          _vp, _vp, C.c_int, _vp]),
    'rz_net_stem_tc': (C.c_int, [_GD, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_net_stem_tc_planes': (C.c_int, [_GD, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_net_stem_go_tc': (C.c_int, [_GD, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_net_stem_go_tc_planes': (C.c_int, [_GD, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'rz_net_conv3x3_f32': (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, _vp]),
    'rz_net_heads': (C.c_int, [C.POINTER(HeadsDesc), _vp, _vp, _vp, C.c_int, _vp]),
    'rz_net_head_features': (C.c_int, [C.POINTER(HeadsDesc), _vp, _vp, C.c_int, _vp]),
    'rz_net_heads_tc': (C.c_int, [C.POINTER(HeadsDesc), _vp, _vp, _vp, C.c_int, _vp]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def row_stride(H, W, requested=0):
    """Row stride S of the padded position layout of the tensor-core network path (rz_row_stride in
    rz_common.cuh): the smallest of 8 / 16 / 20 that leaves a zero column and a zero row, or the explicit
    request; 0 if the board does not fit."""
    m = max(int(H), int(W))
    if requested:
        return int(requested) if requested in (8, 16, 20) and m < requested else 0
    return 8 if m <= 7 else (16 if m <= 15 else (20 if m <= 19 else 0))


def load():
    """Load the shared object (once) and type every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            'rlzero_b200 CUDA library not built: %s is missing. Run `python -m rlzero_b200.build` '
            '(there is no CPU fallback).' % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise NativeLibraryError('symbol %s missing from %s' % (name, LIB_PATH))
        fn.restype = res
        fn.argtypes = args
    if lib.rz_abi_version() != ABI_VERSION:
        raise NativeLibraryError('ABI mismatch: library %d, binding %d (rebuild)' % (
            lib.rz_abi_version(), ABI_VERSION))
    if (lib.rz_sizeof_tree_desc() != C.sizeof(TreeDesc) or lib.rz_sizeof_traj_desc() != C.sizeof(TrajDesc)
            or lib.rz_sizeof_mz_desc() != C.sizeof(MzDesc)):
        raise NativeLibraryError('descriptor struct size mismatch between header and binding')
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        raise NativeLibraryError('%s failed (%d): %s' % (what, rc, load().rz_last_error().decode()))


def ptr(t):
    """Device (or host) address of a torch tensor, None -> NULL."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)
