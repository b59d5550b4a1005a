"""CPU tests: the C-ABI library builds, loads and exports every symbol the header declares
(no compute calls -- there is no GPU here)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    from rlzero_b200 import build
    build.build()
    from rlzero_b200 import _lib
    return _lib.load()


def header_symbols():
    text = open(os.path.join(ROOT, 'include', 'rlzero_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(rz_[a-z0-9_]+)\s*\(', text)))


def test_header_symbols_exported(lib):
    from rlzero_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 16
    for s in syms:
        assert hasattr(lib, s), 'library does not export ' + s
        assert s in _lib.SIGNATURES, 'binding does not type ' + s
    assert sorted(_lib.SIGNATURES) == syms


def test_superseded_convolutions_are_not_exported(lib):
    """Revision 1 of the trunk convolution, its plane encoder and the flag-less fused-heads entry point are gone
    (rz_net_conv3x3_tc2 / rz_net_stem_tc / rz_net_conv3x3_tc2_head_ex do their work)."""
    for s in ('rz_net_conv3x3_tc', 'rz_gomoku_encode_tc', 'rz_net_conv3x3_tc2_head'):
        assert not hasattr(lib, s), s


def test_conv3x3_tc2_rejects_single_cta_groups(lib):
    """rz_net_conv3x3_tc2 runs on CTA pairs only: cta_group 1 is rejected on the host before any launch."""
    dummy = C.c_void_p(16)
    rc = lib.rz_net_conv3x3_tc2(dummy, dummy, dummy, None, C.c_void_p(32), 1, 15, 15, 128, 1, 1, 514, 0, None)
    assert rc != 0 and b'cta_group' in lib.rz_last_error()


def test_abi_version_and_struct_sizes(lib):
    from rlzero_b200 import _lib
    assert lib.rz_abi_version() == _lib.ABI_VERSION
    assert lib.rz_sizeof_tree_desc() == C.sizeof(_lib.TreeDesc)
    assert lib.rz_sizeof_traj_desc() == C.sizeof(_lib.TrajDesc)


def test_argument_errors_are_reported(lib):
    """Argument validation happens on the host before any launch, so it is testable here."""
    from rlzero_b200 import _lib
    g = _lib.GameDesc(40, 5, 1600, 1600)
    rc = lib.rz_gomoku_reset(C.byref(g), None, None, 1, 0, None)
    assert rc != 0 and b'board_size' in lib.rz_last_error()
    g = _lib.GameDesc(15, 5, 225, 230)
    rc = lib.rz_gomoku_step(C.byref(g), None, None, None, None, None, 1, None)
    assert rc != 0 and b'action_stride' in lib.rz_last_error()
    t = _lib.TreeDesc()
    t.game = _lib.GameDesc(15, 5, 225, 256)
    t.n_trees, t.max_nodes, t.max_depth, t.rule = 1, 8, 226, 7
    rc = lib.rz_tree_select(C.byref(t), None)
    assert rc != 0 and b'rule' in lib.rz_last_error()


def test_product_does_not_import_oracle():
    """The product package must never reach into oracle/ (test infrastructure)."""
    for base, _, files in os.walk(os.path.join(ROOT, 'rlzero_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                text = open(os.path.join(base, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', text, flags=re.M), f


def test_no_gpu_means_loud_failure():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from rlzero_b200 import _lib
    from rlzero_b200.engine import SearchForest
    from rlzero_b200.games.gomoku import GomokuEnv
    with pytest.raises(_lib.NativeLibraryError):
        SearchForest(1, 3, 3, n_playout=10)
    with pytest.raises(_lib.NativeLibraryError):
        GomokuEnv(3, 3).reset()


def test_new_entry_points_validate_arguments(lib):
    """Go / DeepMindMCTS / MuZero entry points: host-side validation without a GPU."""
    from rlzero_b200 import _lib
    assert lib.rz_sizeof_mz_desc() == C.sizeof(_lib.MzDesc)
    go = _lib.GameDesc(19, 1, 361, 384, 19, _lib.GAME_GO, 7.5, 0)          # the pass action is missing
    rc = lib.rz_go_reset(C.byref(go), None, None, None, 1, 0, None)
    assert rc != 0 and b'362' in lib.rz_last_error()
    gomoku = _lib.GameDesc(15, 5, 225, 256)
    rc = lib.rz_go_step(C.byref(gomoku), None, None, None, None, None, None, 1, None)
    assert rc != 0 and b'RZ_GAME_GO' in lib.rz_last_error()
    go = _lib.GameDesc(19, 1, 362, 384, 19, _lib.GAME_GO, 7.5, 0)
    rc = lib.rz_gomoku_step(C.byref(go), None, None, None, None, None, 1, None)
    assert rc != 0 and b'rz_go_' in lib.rz_last_error()
    t = _lib.TreeDesc()
    t.game = _lib.GameDesc(15, 5, 225, 256)
    t.n_trees, t.max_nodes, t.max_depth, t.rule, t.flavour = 1, 8, 226, 0, 3
    rc = lib.rz_tree_select(C.byref(t), None)
    assert rc != 0
    m = _lib.MzDesc()
    m.n_trees, m.n_actions, m.action_stride, m.max_nodes, m.max_depth = 1, 225, 230, 51, 51
    rc = lib.rz_mz_select(C.byref(m), None)
    assert rc != 0 and b'action_stride' in lib.rz_last_error()
    rc = lib.rz_mz_gather(None, None, None, None, 1, 15, 15, 16, 256, None)
    assert rc != 0 and b'null' in lib.rz_last_error()


def test_new_host_classes_fail_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from rlzero_b200 import _lib
    from rlzero_b200.games.go import GoBoards, GoEnv
    from rlzero_b200.muzero import MuZeroNet, MuZeroSearch
    with pytest.raises(_lib.NativeLibraryError):
        GoBoards(1, 9)
    with pytest.raises(_lib.NativeLibraryError):
        GoEnv(9).reset()
    with pytest.raises(_lib.NativeLibraryError):
        MuZeroSearch(1, MuZeroNet(6, 0, 0))


def test_row_stride_rule_and_validation(lib):
    """Padded position layout of the network kernels: S = the smallest of 8 / 16 / 20 above max(H, W) (ABI 7);
    the Python mirror and the C validation agree."""
    from rlzero_b200 import _lib as L
    assert [L.row_stride(h, w) for h, w in [(3, 3), (6, 7), (7, 7), (8, 8), (6, 8), (15, 15), (16, 16), (19, 19)]] == \
        [8, 8, 8, 16, 16, 16, 20, 20]
    assert L.row_stride(20, 20) == 0 and L.row_stride(9, 9, 8) == 0 and L.row_stride(6, 7, 16) == 16
    g = L.GameDesc(6, 4, 7, 32, 7, L.GAME_CONNECT4, 0.0, 0, 12)
    rc = lib.rz_gomoku_reset(C.byref(g), None, None, 1, 0, None)
    assert rc != 0 and b'row_stride' in lib.rz_last_error()
    # a 9x9 board does not fit the 8-stride layout: rejected on the host before any launch
    g = L.GameDesc(9, 5, 81, 96, 9, L.GAME_GOMOKU, 0.0, 0, 8)
    dummy = C.c_void_p(16)
    rc = lib.rz_net_stem_tc(C.byref(g), dummy, dummy, dummy, dummy, dummy, 1, 1, 0, None)
    assert rc != 0 and b'row_stride' in lib.rz_last_error()
    rc = lib.rz_net_conv3x3_tc3(dummy, dummy, dummy, None, C.c_void_p(32), 1, 6, 7, 12, 1, 0, None)
    assert rc != 0 and b'row_stride' in lib.rz_last_error()


def test_leaf_parallel_descriptor_is_validated(lib):
    """rz_tree_desc.leaves_per_tree > 1 needs its scratch and the AlphaZero flavour (host-side validation)."""
    from rlzero_b200 import _lib
    t = _lib.TreeDesc()
    t.game = _lib.GameDesc(15, 5, 225, 256)
    t.n_trees, t.max_nodes, t.max_depth, t.rule, t.ln_table_len = 1, 8, 226, 0, 16
    dummy = 64
    for name in ('edge_N', 'edge_W', 'edge_child', 'node_parent', 'node_paction', 'n_nodes', 'root_N', 'root_W',
                 'root_rows', 'root_meta', 'path_node', 'path_action', 'depth', 'leaf_rows', 'leaf_meta', 'ln_table'):
        setattr(t, name, dummy)
    t.leaves_per_tree = 4
    rc = lib.rz_tree_select(C.byref(t), None)
    assert rc != 0 and b'vl_saved_W' in lib.rz_last_error()
    t.leaves_per_tree = 1000
    rc = lib.rz_tree_select(C.byref(t), None)
    assert rc != 0 and b'leaves_per_tree' in lib.rz_last_error()
    t.leaves_per_tree, t.vl_saved_W, t.flavour, t.edge_O, t.root_O = 4, dummy, _lib.FLAVOUR_DEEPMIND, dummy, dummy
    rc = lib.rz_tree_select(C.byref(t), None)
    assert rc != 0 and b'AlphaZero flavour' in lib.rz_last_error()
