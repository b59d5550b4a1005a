"""CPU tests of the training entry points for the 20-stride layout and the 17-plane Go stem: argument validation on the
host (before any launch, so no GPU is needed) and which modules get a native trainer."""
import ctypes as C

import pytest


@pytest.fixture(scope='module')
def lib():
    from rlzero_b200 import build
    build.build()
    from rlzero_b200 import _lib
    return _lib.load()


def _err(lib):
    return lib.rz_last_error()


def test_ex_entry_points_reject_a_bad_row_stride(lib):
    d = C.c_void_p(256)
    for S in (0, 8, 15, 19, 24):
        calls = [
            lambda: lib.rz_learn_conv_wgrad_tc_ex(d, d, d, d, 1 << 30, 4, S, 0, None),
            lambda: lib.rz_learn_bn_forward_ex(d, None, d, d, d, None, None, 1e-5, 0.1, d, d, 4, 9, 9, S, None),
            lambda: lib.rz_learn_bn_backward_ex(d, d, d, d, d, d, d, None, d, 4, 9, 9, S, None),
            lambda: lib.rz_learn_relu_bwd_bf16_ex(d, d, d, 4, S, None),
            lambda: lib.rz_learn_tile_colsum_ex(d, d, d, 4, S, None),
            lambda: lib.rz_learn_tile_to_nhwc_ex(d, d, 4, 9, 9, S, None),
            lambda: lib.rz_learn_nhwc_to_tile_ex(d, d, 4, 9, 9, S, None),
            lambda: lib.rz_learn_planes_to_tile_ex(d, 17, d, 4, 9, 9, S, None),
        ]
        for call in calls:
            assert call() != 0 and b'row_stride' in _err(lib), (S, _err(lib))


def test_ex_entry_points_reject_a_board_that_does_not_fit(lib):
    d = C.c_void_p(256)
    for H, W, S in ((16, 16, 16), (20, 20, 20), (19, 21, 20), (0, 9, 16), (9, 0, 20)):
        calls = [
            lambda: lib.rz_learn_bn_forward_ex(d, None, d, d, d, None, None, 1e-5, 0.1, d, d, 4, H, W, S, None),
            lambda: lib.rz_learn_bn_backward_ex(d, d, d, d, d, d, d, None, d, 4, H, W, S, None),
            lambda: lib.rz_learn_tile_to_nhwc_ex(d, d, 4, H, W, S, None),
            lambda: lib.rz_learn_nhwc_to_tile_ex(d, d, 4, H, W, S, None),
            lambda: lib.rz_learn_planes_to_tile_ex(d, 4, d, 4, H, W, S, None),
        ]
        for call in calls:
            assert call() != 0 and b'board' in _err(lib), (H, W, S, _err(lib))
    # the 16-stride entry points keep their 15x15 limit
    assert lib.rz_learn_bn_forward(d, None, d, d, d, None, None, 1e-5, 0.1, d, d, 4, 19, 19, None) != 0
    assert b'board' in _err(lib)


def test_ex_entry_points_reject_bad_plane_counts(lib):
    d = C.c_void_p(256)
    for P in (0, 3, 5, 16, 18):
        assert lib.rz_learn_planes_to_tile_ex(d, P, d, 4, 19, 19, 20, None) != 0 and b'n_planes' in _err(lib)
        assert lib.rz_learn_pack_stem_tc_ex(d, P, d, None) != 0 and b'in_planes' in _err(lib)


def test_which_resnets_get_a_native_trainer():
    """make_trainer: the default keeps Go networks and 16x16 .. 19x19 boards on autograd (None); asked for, they get
    ResNetTrainer (which needs a GPU, so here the request fails loudly instead of falling back).  Rectangular boards and
    other plane / action counts get no native trainer either way."""
    import torch
    from rlzero_b200 import _lib
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    from rlzero_b200.learn import make_trainer, resnet_trainer_fits
    go19 = ResNetPolicyValueNet(19, n_blocks=1, n_actions=362, in_planes=17)
    go9 = ResNetPolicyValueNet(9, n_blocks=1, n_actions=82, in_planes=17)
    gomoku17 = ResNetPolicyValueNet(17, n_blocks=1)
    for net in (go19, go9, gomoku17):
        assert resnet_trainer_fits(net)
        assert make_trainer(net) is None
    c4 = ResNetPolicyValueNet(6, n_blocks=1, board_width=7, n_actions=7)
    odd = [c4, ResNetPolicyValueNet(9, n_blocks=1, in_planes=8), ResNetPolicyValueNet(9, n_blocks=1, n_actions=82),
           ResNetPolicyValueNet(9, n_blocks=1, n_actions=81, in_planes=17)]
    for net in odd:
        assert not resnet_trainer_fits(net)
        assert make_trainer(net, requested=True) is None
    if not torch.cuda.is_available():
        with pytest.raises(_lib.NativeLibraryError):
            make_trainer(go19, requested=True)
