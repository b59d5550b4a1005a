"""TEST INFRASTRUCTURE ONLY -- builds oracle/c/rz_oracle.c (the plain-C restatement of the reference
search) into oracle/_build/librz_oracle.so with gcc, and loads it through ctypes.

    python -m oracle.build_oracle

The shared object is git-ignored and travels to the GPU box with the repository snapshot; building
the checker is not using it: only tests/ load it."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'c', 'rz_oracle.c')
SRC_GO = os.path.join(HERE, 'c', 'rz_go_oracle.c')      # Go rules + search (config 4), same shared object
OUT_DIR = os.path.join(HERE, '_build')
LIB = os.path.join(OUT_DIR, 'librz_oracle.so')


def build(force=False):
    if (not force and os.path.exists(LIB) and os.path.getmtime(LIB) > os.path.getmtime(SRC)
            and os.path.getmtime(LIB) > os.path.getmtime(SRC_GO)):
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    cmd = ['gcc', '-O2', '-ffp-contract=off', '-fopenmp', '-shared', '-fPIC', '-o', LIB + '.tmp', SRC, SRC_GO, '-lm']
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if out.returncode != 0:
        raise RuntimeError('gcc failed:\n' + out.stdout.decode())
    os.replace(LIB + '.tmp', LIB)
    return LIB


_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        lib = C.CDLL(LIB)
        i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
        lib.rzo_search_game.restype = C.c_int
        lib.rzo_search_game.argtypes = [C.c_int, C.c_int, i32p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                                        C.c_int, i32p, i32p, f64p, i32p, f64p]
        lib.rzo_search_batch.restype = C.c_int
        lib.rzo_search_batch.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_double,
                                         C.c_int, C.c_int, i32p, f64p, i32p, f64p]
        lib.rzo_search_batch_vl.restype = C.c_int
        lib.rzo_search_batch_vl.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_double,
                                            C.c_int, C.c_int, C.c_int, C.c_double, i32p, f64p, i32p, f64p]
        lib.rzo_search_batch_c4.restype = C.c_int
        lib.rzo_search_batch_c4.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_double,
                                            C.c_int, C.c_int, C.c_int, C.c_double, i32p, f64p, i32p, f64p]
        lib.rzo_replay_games.restype = C.c_int
        lib.rzo_replay_games.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, i32p, i32p, i32p]
        lib.rzo_search_batch_reuse.restype = C.c_int
        lib.rzo_search_batch_reuse.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_double,
                                               C.c_int, C.c_int, i32p, i32p, f64p, i32p, f64p]
        lib.rzo_dm_search_batch.restype = C.c_int
        lib.rzo_dm_search_batch.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_double, C.c_int,
                                            C.c_int, C.c_int, C.c_int, i32p, f64p, i32p, i32p, f64p, i32p, i32p]
        i8p = C.POINTER(C.c_int8)
        lib.rzo_go_search_batch.restype = C.c_int
        lib.rzo_go_search_batch.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_double,
                                            C.c_int, C.c_int, i32p, f64p, i32p, f64p]
        lib.rzo_go_random_games.restype = C.c_int
        lib.rzo_go_random_games.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int, i32p, C.c_int, C.c_uint64, i32p, i32p,
                                            i8p, i32p, i32p, i32p, f64p, i8p]
        lib.rzo_philox4.restype = None
        lib.rzo_philox4.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32)]
        lib.rzo_go_rollout_dm.restype = C.c_int
        lib.rzo_go_rollout_dm.argtypes = [C.c_int, C.c_double, C.c_int, i8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, f64p, i8p]
        _lib = lib
    return _lib


def search_game(size, k, moves, n_playout, cpuct=5.0, rule=0, eval_id=2, follow=()):
    """Search a position (after ``moves``), then again after each move of ``follow`` with the subtree
    kept.  Returns (visits [n,A] int32, W [n,A] float64, root_N [n], root_W [n])."""
    import numpy as np
    lib = load()
    A = size * size
    n = len(follow) + 1
    mv = np.ascontiguousarray(np.asarray(list(moves) + [0], dtype=np.int32))
    fl = np.ascontiguousarray(np.asarray(list(follow) + [0], dtype=np.int32))
    visits = np.zeros((n, A), dtype=np.int32)
    w = np.zeros((n, A), dtype=np.float64)
    rn = np.zeros(n, dtype=np.int32)
    rw = np.zeros(n, dtype=np.float64)
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_search_game(size, k, mv.ctypes.data_as(i32p), len(moves), n_playout, float(cpuct), int(rule),
                             int(eval_id), n, fl.ctypes.data_as(i32p), visits.ctypes.data_as(i32p),
                             w.ctypes.data_as(f64p), rn.ctypes.data_as(i32p), rw.ctypes.data_as(f64p))
    if rc:
        raise RuntimeError('rzo_search_game failed (%d)' % rc)
    return visits, w, rn, rw


def search_batch(size, k, move_lists, n_playout, cpuct=5.0, rule=0, eval_id=2):
    """One fresh search per game, all host cores.  Returns (visits [G,A], W [G,A], root_N [G], root_W [G])."""
    import numpy as np
    lib = load()
    G, A = len(move_lists), size * size
    mx = max(1, max((len(m) for m in move_lists), default=0))
    mv = np.zeros((G, mx), dtype=np.int32)
    nm = np.zeros(G, dtype=np.int32)
    for g, m in enumerate(move_lists):
        mv[g, :len(m)] = m
        nm[g] = len(m)
    visits = np.zeros((G, A), dtype=np.int32)
    w = np.zeros((G, A), dtype=np.float64)
    rn = np.zeros(G, dtype=np.int32)
    rw = np.zeros(G, dtype=np.float64)
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_search_batch(G, size, k, mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), mx, n_playout,
                              float(cpuct), int(rule), int(eval_id), visits.ctypes.data_as(i32p),
                              w.ctypes.data_as(f64p), rn.ctypes.data_as(i32p), rw.ctypes.data_as(f64p))
    if rc:
        raise RuntimeError('rzo_search_batch failed (%d)' % rc)
    return visits, w, rn, rw


def search_batch_vl(size, k, move_lists, n_playout, cpuct=5.0, rule=0, eval_id=2, leaves_per_wave=8, virtual_loss=1.0):
    """``search_batch`` in the product's leaf-parallel mode (waves of up to ``leaves_per_wave`` playouts with virtual
    loss; parity unpinned: the reference has no such mode)."""
    import numpy as np
    lib = load()
    G, A = len(move_lists), size * size
    mx = max(1, max((len(m) for m in move_lists), default=0))
    mv = np.zeros((G, mx), dtype=np.int32)
    nm = np.zeros(G, dtype=np.int32)
    for g, m in enumerate(move_lists):
        mv[g, :len(m)] = m
        nm[g] = len(m)
    visits = np.zeros((G, A), dtype=np.int32)
    w = np.zeros((G, A), dtype=np.float64)
    rn = np.zeros(G, dtype=np.int32)
    rw = np.zeros(G, dtype=np.float64)
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_search_batch_vl(G, size, k, mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), mx, n_playout,
                                 float(cpuct), int(rule), int(eval_id), int(leaves_per_wave), float(virtual_loss),
                                 visits.ctypes.data_as(i32p), w.ctypes.data_as(f64p), rn.ctypes.data_as(i32p),
                                 rw.ctypes.data_as(f64p))
    if rc:
        raise RuntimeError('rzo_search_batch_vl failed (%d)' % rc)
    return visits, w, rn, rw


def search_batch_c4(move_lists, n_playout, cpuct=5.0, rule=0, eval_id=2, rows=6, cols=7, k=4, leaves_per_wave=1,
                    virtual_loss=1.0):
    """Connect Four (actions = columns): one fresh search per game; ``leaves_per_wave = 1`` is the reference's
    sequential search over that game.  Returns (visits [G,cols], W [G,cols], root_N [G], root_W [G])."""
    import numpy as np
    lib = load()
    G = len(move_lists)
    mx = max(1, max((len(m) for m in move_lists), default=0))
    mv = np.zeros((G, mx), dtype=np.int32)
    nm = np.zeros(G, dtype=np.int32)
    for g, m in enumerate(move_lists):
        mv[g, :len(m)] = m
        nm[g] = len(m)
    visits = np.zeros((G, cols), dtype=np.int32)
    w = np.zeros((G, cols), dtype=np.float64)
    rn = np.zeros(G, dtype=np.int32)
    rw = np.zeros(G, dtype=np.float64)
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_search_batch_c4(G, rows, cols, k, mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), mx, n_playout,
                                 float(cpuct), int(rule), int(eval_id), int(leaves_per_wave), float(virtual_loss),
                                 visits.ctypes.data_as(i32p), w.ctypes.data_as(f64p), rn.ctypes.data_as(i32p),
                                 rw.ctypes.data_as(f64p))
    if rc:
        raise RuntimeError('rzo_search_batch_c4 failed (%d)' % rc)
    return visits, w, rn, rw


def replay_games(size, k, moves):
    """GomokuEnv.step until game_end_winner for every row of ``moves`` [G, T] (int32).  Returns (end_ply, winner,
    ended) int32 [G]."""
    import numpy as np
    lib = load()
    mv = np.ascontiguousarray(moves, dtype=np.int32)
    G, T = mv.shape
    nm = np.full(G, T, dtype=np.int32)
    end_ply, winner, ended = (np.zeros(G, dtype=np.int32) for _ in range(3))
    i32p = C.POINTER(C.c_int32)
    rc = lib.rzo_replay_games(G, size, k, mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), T,
                              end_ply.ctypes.data_as(i32p), winner.ctypes.data_as(i32p), ended.ctypes.data_as(i32p))
    if rc:
        raise RuntimeError('rzo_replay_games failed (%d)' % rc)
    return end_ply, winner, ended


def search_batch_reuse(size, k, move_lists, n_playout, cpuct=5.0, rule=0, eval_id=2):
    """Search, play the most visited move (lowest action on ties), search again with the subtree kept
    (update_with_move).  Returns (move [G], visits [G,A], W [G,A], root_N [G], root_W [G]) of the SECOND search;
    games that the move ends report zeros."""
    import numpy as np
    lib = load()
    G, A = len(move_lists), size * size
    mx = max(1, max((len(m) for m in move_lists), default=0))
    mv = np.zeros((G, mx), dtype=np.int32)
    nm = np.zeros(G, dtype=np.int32)
    for g, m in enumerate(move_lists):
        mv[g, :len(m)] = m
        nm[g] = len(m)
    move = np.zeros(G, dtype=np.int32)
    visits = np.zeros((G, A), dtype=np.int32)
    w = np.zeros((G, A), dtype=np.float64)
    rn = np.zeros(G, dtype=np.int32)
    rw = np.zeros(G, dtype=np.float64)
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_search_batch_reuse(G, size, k, mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), mx, n_playout,
                                    float(cpuct), int(rule), int(eval_id), move.ctypes.data_as(i32p),
                                    visits.ctypes.data_as(i32p), w.ctypes.data_as(f64p), rn.ctypes.data_as(i32p),
                                    rw.ctypes.data_as(f64p))
    if rc:
        raise RuntimeError('rzo_search_batch_reuse failed (%d)' % rc)
    return move, visits, w, rn, rw


def dm_search_batch(size, k, move_lists, sims, uct_c=2.0, method='puct', solve=True, returns_mode=0, eval_id=2):
    """The reference's DeepMindMCTS (no shuffle, no noise) on every position.  Returns a dict of arrays: visits [G,A]
    (-1 = not a root child), w [G,A], outcome [G,A] (0 none, else 0x100 | (o0+1) | (o1+1) << 2), root_n, root_w,
    root_outcome, best [G]."""
    import numpy as np
    lib = load()
    G, A = len(move_lists), size * size
    mx = max(1, max((len(m) for m in move_lists), default=0))
    mv = np.zeros((G, mx), dtype=np.int32)
    nm = np.zeros(G, dtype=np.int32)
    for g, m in enumerate(move_lists):
        mv[g, :len(m)] = m
        nm[g] = len(m)
    out = dict(visits=np.zeros((G, A), dtype=np.int32), w=np.zeros((G, A), dtype=np.float64),
               outcome=np.zeros((G, A), dtype=np.int32), root_n=np.zeros(G, dtype=np.int32),
               root_w=np.zeros(G, dtype=np.float64), root_outcome=np.zeros(G, dtype=np.int32),
               best=np.zeros(G, dtype=np.int32))
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_dm_search_batch(G, size, k, mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), mx, int(sims),
                                 float(uct_c), 1 if method == 'puct' else 0, int(bool(solve)), int(returns_mode),
                                 int(eval_id), out['visits'].ctypes.data_as(i32p), out['w'].ctypes.data_as(f64p),
                                 out['outcome'].ctypes.data_as(i32p), out['root_n'].ctypes.data_as(i32p),
                                 out['root_w'].ctypes.data_as(f64p), out['root_outcome'].ctypes.data_as(i32p),
                                 out['best'].ctypes.data_as(i32p))
    if rc:
        raise RuntimeError('rzo_dm_search_batch failed (%d)' % rc)
    return out


if __name__ == '__main__':
    print(build(force=True))


def go_search_batch(n, move_lists, n_playout, komi=7.5, move_cap=0, cpuct=5.0, rule=0, eval_id=2):
    """One fresh AlphaZero search per Go position (oracle/c/rz_go_oracle.c), all host cores.
    Returns (visits [G, n*n+1], W, root_N, root_W)."""
    import numpy as np
    lib = load()
    G, A = len(move_lists), n * n + 1
    mx = max(1, max((len(m) for m in move_lists), default=0))
    mv = np.zeros((G, mx), dtype=np.int32)
    nm = np.zeros(G, dtype=np.int32)
    for g, m in enumerate(move_lists):
        mv[g, :len(m)] = m
        nm[g] = len(m)
    visits = np.zeros((G, A), dtype=np.int32)
    w = np.zeros((G, A), dtype=np.float64)
    rn = np.zeros(G, dtype=np.int32)
    rw = np.zeros(G, dtype=np.float64)
    i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    rc = lib.rzo_go_search_batch(G, n, float(komi), int(move_cap), mv.ctypes.data_as(i32p), nm.ctypes.data_as(i32p), mx,
                                 n_playout, float(cpuct), int(rule), int(eval_id), visits.ctypes.data_as(i32p),
                                 w.ctypes.data_as(f64p), rn.ctypes.data_as(i32p), rw.ctypes.data_as(f64p))
    if rc:
        raise RuntimeError('rzo_go_search_batch failed (%d)' % rc)
    return visits, w, rn, rw


def go_random_games(G, n, n_plies, komi=7.5, move_cap=0, seed=1):
    """Random legal Go games by the C oracle's rules: dict(moves [G, max], played [G], cell [G, n*n] (+1 black, -1
    white), ko, to_play (0 black), over, score float64, legal [G, n*n+1])."""
    import numpy as np
    lib = load()
    plies = np.ascontiguousarray(np.broadcast_to(np.asarray(n_plies, dtype=np.int32), (G,)))
    mx = max(1, int(plies.max()))
    out = dict(moves=np.zeros((G, mx), dtype=np.int32), played=np.zeros(G, dtype=np.int32),
               cell=np.zeros((G, n * n), dtype=np.int8), ko=np.zeros(G, dtype=np.int32),
               to_play=np.zeros(G, dtype=np.int32), over=np.zeros(G, dtype=np.int32),
               score=np.zeros(G, dtype=np.float64), legal=np.zeros((G, n * n + 1), dtype=np.int8))
    i32p, f64p, i8p = C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_int8)
    rc = lib.rzo_go_random_games(G, n, float(komi), int(move_cap), plies.ctypes.data_as(i32p), mx, int(seed),
                                 out['moves'].ctypes.data_as(i32p), out['played'].ctypes.data_as(i32p),
                                 out['cell'].ctypes.data_as(i8p), out['ko'].ctypes.data_as(i32p),
                                 out['to_play'].ctypes.data_as(i32p), out['over'].ctypes.data_as(i32p),
                                 out['score'].ctypes.data_as(f64p), out['legal'].ctypes.data_as(i8p))
    if rc:
        raise RuntimeError('rzo_go_random_games failed (%d)' % rc)
    return out
