"""CPU tests of the batched one-launch trunk's entry point (rz_net_trunk_tc2): exported, typed, and its arguments checked
on the host before any launch."""
import ctypes as C

import pytest


@pytest.fixture(scope='module')
def lib():
    from rlzero_b200 import build
    build.build()
    from rlzero_b200 import _lib
    return _lib.load()


def test_batched_trunk_is_exported_at_abi_14(lib):
    from rlzero_b200 import _lib
    assert _lib.ABI_VERSION == 14 and lib.rz_abi_version() == 14
    assert hasattr(lib, 'rz_net_trunk_tc2') and 'rz_net_trunk_tc2' in _lib.SIGNATURES


@pytest.mark.parametrize('change,needle', [
    (dict(act_in=None), b'act_in'), (dict(weights=None), b'weights'), (dict(biases=None), b'biases_host'),
    (dict(scratch=None), b'scratch'), (dict(feat=None), b'feat'), (dict(w1x1=None), b'w1x1'),
    (dict(n_layers=0), b'n_layers'), (dict(n_layers=25), b'n_layers'), (dict(res_mask=1), b'res_mask'),
    (dict(res_mask=1 << 20), b'res_mask'), (dict(chunk=0), b'chunk'), (dict(chunk=17), b'chunk'),
    (dict(n_boards=-1), b'n_boards'), (dict(H=16), b'board_size'), (dict(W=0), b'board_cols'),
    (dict(n_ctas=1), b'n_ctas'), (dict(n_ctas=-2), b'n_ctas')])
def test_batched_trunk_rejects_bad_arguments(lib, change, needle):
    dummy = C.c_void_p(256)
    host = (C.c_float * (24 * 128))()
    a = dict(act_in=dummy, weights=dummy, biases=C.cast(host, C.c_void_p), n_layers=20, relu_mask=(1 << 20) - 1,
             res_mask=0xAAAAA, scratch=dummy, chunk=8, n_boards=8192, H=15, W=15, w1x1=C.cast(host, C.c_void_p),
             b1x1=C.cast(host, C.c_void_p), feat=dummy, n_ctas=0)
    a.update(change)
    rc = lib.rz_net_trunk_tc2(a['act_in'], a['weights'], a['biases'], a['n_layers'], a['relu_mask'], a['res_mask'],
                              a['scratch'], a['chunk'], a['n_boards'], a['H'], a['W'], a['w1x1'], a['b1x1'], a['feat'],
                              a['n_ctas'], None)
    assert rc != 0 and needle in lib.rz_last_error(), lib.rz_last_error()
