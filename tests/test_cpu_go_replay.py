"""CPU tests of the Go training-record entry points (rz_go_records_pack / rz_go_records_expand): exported and typed,
every argument checked on the host before any launch, and rz_augment_equi limited to square Gomoku boards."""
import ctypes as C

import pytest


@pytest.fixture(scope='module')
def lib():
    from rlzero_b200 import build
    build.build()
    from rlzero_b200 import _lib
    return _lib.load()


def _go(H=9):
    from rlzero_b200 import _lib as L
    A = H * H + 1
    return L.GameDesc(H, 1, A, (A + 31) // 32 * 32, H, L.GAME_GO, 7.5, 0)


D = C.c_void_p(64)       # never dereferenced: every call below fails its host-side checks


def _pack(lib, g, rows=D, info=D, info_stride=6, pi=D, n=4, planes=D, mover=D, out_pi=D, z=D, capacity=8, dst_start=0):
    return lib.rz_go_records_pack(C.byref(g), rows, info, info_stride, pi, n, planes, mover, out_pi, z, capacity,
                                  dst_start, None)


def _expand(lib, g, planes=D, mover=D, pi=D, z=D, capacity=8, slots=D, syms=D, n=4, out_states=D, out_pi=D, out_z=D):
    return lib.rz_go_records_expand(C.byref(g), planes, mover, pi, z, capacity, slots, syms, n, out_states, out_pi,
                                    out_z, None)


def test_go_record_symbols_are_exported_and_typed(lib):
    from rlzero_b200 import _lib as L
    for s in ('rz_go_records_pack', 'rz_go_records_expand'):
        assert hasattr(lib, s) and s in L.SIGNATURES
        assert getattr(lib, s).argtypes == L.SIGNATURES[s][1]


@pytest.mark.parametrize('kw,word', [
    (dict(rows=None), b'rows'), (dict(info=None), b'info'), (dict(pi=None), b'pi'), (dict(planes=None), b'planes'),
    (dict(mover=None), b'mover'), (dict(out_pi=None), b'out_pi'), (dict(z=None), b'z'), (dict(n=-1), b'n -1'),
    (dict(info_stride=5), b'info_stride'), (dict(capacity=0), b'capacity'), (dict(dst_start=8), b'dst_start'),
    (dict(dst_start=-1), b'dst_start')])
def test_pack_rejects_bad_arguments(lib, kw, word):
    rc = _pack(lib, _go(), **kw)
    assert rc != 0 and word in lib.rz_last_error(), lib.rz_last_error()


@pytest.mark.parametrize('kw,word', [
    (dict(planes=None), b'planes'), (dict(mover=None), b'mover'), (dict(pi=None), b'pi'), (dict(z=None), b'z'),
    (dict(slots=None), b'slots'), (dict(syms=None), b'syms'), (dict(out_states=None), b'out_states'),
    (dict(out_pi=None), b'out_pi'), (dict(out_z=None), b'out_z'), (dict(n=-3), b'n -3'), (dict(capacity=0), b'capacity')])
def test_expand_rejects_bad_arguments(lib, kw, word):
    rc = _expand(lib, _go(), **kw)
    assert rc != 0 and word in lib.rz_last_error(), lib.rz_last_error()


def test_go_record_entry_points_need_a_go_descriptor(lib):
    from rlzero_b200 import _lib as L
    gomoku = L.GameDesc(9, 5, 81, 96)
    for call in (_pack, _expand):
        rc = call(lib, gomoku)
        assert rc != 0 and b'RZ_GAME_GO' in lib.rz_last_error()
    no_pass = L.GameDesc(9, 1, 81, 96, 9, L.GAME_GO, 7.5, 0)
    rc = _pack(lib, no_pass)
    assert rc != 0 and b'82' in lib.rz_last_error()


def test_augment_equi_takes_square_gomoku_only(lib):
    """rz_augment_equi knows the 4-plane Gomoku encoding on square boards: Go, Connect Four and rectangular Gomoku are
    rejected on the host, Go with a pointer to the Go record entry points."""
    from rlzero_b200 import _lib as L
    cases = [(_go(19), b'game_type'), (_go(9), b'rz_go_records'),
             (L.GameDesc(6, 4, 7, 32, 7, L.GAME_CONNECT4, 0.0, 0), b'game_type'),
             (L.GameDesc(6, 4, 42, 64, 7, L.GAME_GOMOKU, 0.0, 0), b'width')]
    for g, word in cases:
        rc = lib.rz_augment_equi(C.byref(g), D, D, 6, D, D, D, D, 4, None)
        assert rc != 0 and word in lib.rz_last_error(), (g.game_type, lib.rz_last_error())
    # square Gomoku, with the width given or left at 0, passes the descriptor checks (and stops at the null output)
    for g in (L.GameDesc(15, 5, 225, 256), L.GameDesc(15, 5, 225, 256, 15, L.GAME_GOMOKU, 0.0, 0)):
        rc = lib.rz_augment_equi(C.byref(g), D, D, 6, D, None, D, D, 4, None)
        assert rc != 0 and b'null argument' in lib.rz_last_error()


def test_go_replay_buffer_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from rlzero_b200 import _lib as L
    from rlzero_b200.train_pipeline import GoReplayBuffer
    with pytest.raises(L.NativeLibraryError):
        GoReplayBuffer(16, 9)
