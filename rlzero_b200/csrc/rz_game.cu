// rlzero_b200 -- batched GomokuEnv kernels (one warp per game) and closed-form evaluators.
// Reference: rlzero/games/gomoku/gomoku_env.py (reset 33-47, step 49-70, leagel_actions 72-73,
// current_state 95-114, has_a_winner 116-170, game_end_winner 196-203).
#include "rz_board.cuh"
#include "rz_go.cuh"

#define RZ_GAME_WARPS 4
#define RZ_GAME_THREADS (RZ_GAME_WARPS * 32)

__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_gomoku_reset_kernel(rz_game_desc gd, uint32_t* rows, int32_t* meta, int n, int only_ended) {
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const int lane = rz_lane(), H = gd.board_size;
  int32_t* m = meta + (size_t)g * RZ_META_STRIDE;
  const int st = m[RZ_META_STATUS];
  if (only_ended && !(st == RZ_ENDED_WIN || st == RZ_ENDED_TIE)) return;
  if (lane < H) { rows[(size_t)g * 2 * H + lane] = 0u; rows[(size_t)g * 2 * H + H + lane] = 0u; }
  if (lane == 0) {
    m[RZ_META_PLAYER] = 0;
    m[RZ_META_LAST_MOVE] = -1;
    m[RZ_META_STONES] = 0;
    m[RZ_META_STATUS] = RZ_ACTIVE;
    m[RZ_META_WINNER] = -1;
    m[RZ_META_PLY] = 0;
    m[RZ_META_FAULT] = 0;
    m[RZ_META_EPISODE] = only_ended ? m[RZ_META_EPISODE] + 1 : 0;
  }
}

__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_gomoku_step_kernel(rz_game_desc gd, uint32_t* rows, int32_t* meta, const int32_t* actions,
                      int32_t* reward, int32_t* win, int n) {
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size;
  const int a = actions[g];
  if (a < 0) return;
  int32_t* m = meta + (size_t)g * RZ_META_STRIDE;
  rz_wboard b;
  rz_board_load(b, rows + (size_t)g * 2 * H, m, H);
  if (a >= gd.n_actions || rz_board_occupied(b, a, q)) {  // gomoku_env.py:51
    if (lane == 0) m[RZ_META_FAULT] |= RZ_FAULT_ILLEGAL_MOVE;
    return;
  }
  const int mover = b.player;
  rz_board_play(b, a, q);
  int winner;
  const int status = rz_board_status(b, q, winner);
  rz_board_store_rows(b, rows + (size_t)g * 2 * H, H);
  if (lane == 0) {
    m[RZ_META_PLAYER] = b.player;
    m[RZ_META_LAST_MOVE] = b.last_move;
    m[RZ_META_STONES] = b.stones;
    m[RZ_META_STATUS] = status;
    m[RZ_META_WINNER] = winner;
    m[RZ_META_PLY] += 1;
    const int w = status == RZ_ENDED_WIN;                   // gomoku_env.py:59-65
    if (win) win[g] = w;
    if (reward) reward[g] = w ? (winner == mover ? 1 : -1) : 0;
  }
}

__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_gomoku_legal_kernel(rz_game_desc gd, const uint32_t* rows, uint8_t* mask, int n) {
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size, A = gd.n_actions;
  const uint32_t occ = lane < H ? (rows[(size_t)g * 2 * H + lane] | rows[(size_t)g * 2 * H + H + lane]) : 0u;
  for (int s0 = 0; s0 < A; s0 += 32) {
    const int s = s0 + lane;
    const bool legal = rz_occ_slot_legal(occ, s, q);
    if (s < A) mask[(size_t)g * A + s] = legal ? 1 : 0;
  }
}

__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_gomoku_winner_kernel(rz_game_desc gd, const uint32_t* rows, const int32_t* meta, int32_t* end,
                        int32_t* winner_out, int n) {
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const int H = gd.board_size;
  rz_wboard b;
  rz_board_load(b, rows + (size_t)g * 2 * H, meta + (size_t)g * RZ_META_STRIDE, H);
  int winner;
  const int status = rz_board_status(b, rz_geom_of(gd), winner);
  if (rz_lane() == 0) {
    end[g] = status != RZ_ACTIVE;
    winner_out[g] = winner;
  }
}

// plane value for (plane, r, c) from the distributed rows -- gomoku_env.py:95-114
__device__ __forceinline__ float rz_plane_value(const rz_wboard& b, uint32_t mine, uint32_t theirs,
                                                int plane, int r, int c, int W) {
  // all lanes call (shuffles inside)
  const uint32_t mrow = __shfl_sync(RZ_FULL, mine, r);
  const uint32_t trow = __shfl_sync(RZ_FULL, theirs, r);
  float v = 0.0f;
  if (plane == 0) v = (float)((mrow >> c) & 1u);
  else if (plane == 1) v = (float)((trow >> c) & 1u);
  else if (plane == 2) v = (b.stones > 0 && b.last_move == r * W + c) ? 1.0f : 0.0f;
  else v = (b.stones & 1) ? 0.0f : 1.0f;
  return v;
}

__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_gomoku_encode_f32_kernel(rz_game_desc gd, const uint32_t* rows, const int32_t* meta,
                            float* planes, int n) {
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size, A = q.cells, W = q.W;
  rz_wboard b;
  rz_board_load(b, rows + (size_t)g * 2 * H, meta + (size_t)g * RZ_META_STRIDE, H);
  const uint32_t mine = b.p[b.player], theirs = b.p[b.player ^ 1];
  const int total = 4 * A;
  for (int i0 = 0; i0 < total; i0 += 32) {
    const int i = i0 + lane;
    const int ic = i < total ? i : 0;
    const int plane = ic / A, pos = ic - plane * A;
    const int r = pos / W, c = pos - r * W;
    const float v = rz_plane_value(b, mine, theirs, plane, r, c, W);
    if (i < total) planes[(size_t)g * total + i] = v;
  }
}

// channels-last float32 [n][HW][4] for the fp32 trunk
__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_gomoku_encode_nhwc_kernel(rz_game_desc gd, const uint32_t* rows, const int32_t* meta,
                             float* planes, int n) {
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size, A = q.cells, W = q.W;
  rz_wboard b;
  rz_board_load(b, rows + (size_t)g * 2 * H, meta + (size_t)g * RZ_META_STRIDE, H);
  const uint32_t mine = b.p[b.player], theirs = b.p[b.player ^ 1];
  const int total = 4 * A;
  for (int i0 = 0; i0 < total; i0 += 32) {
    const int i = i0 + lane;
    const int ic = i < total ? i : 0;
    const int pos = ic >> 2, plane = ic & 3;
    const int r = pos / W, c = pos - r * W;
    const float v = rz_plane_value(b, mine, theirs, plane, r, c, W);
    if (i < total) planes[(size_t)g * total + i] = v;
  }
}

// closed-form evaluators (oracle/evaluators.py) on the leaf positions of a wave
template <class GM>
__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_eval_closed_form_kernel(rz_tree_desc t, int eval_id, float* prior, float* value) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);     // a leaf slot (tree*K + k in leaf-parallel mode)
  if (g >= t.n_trees * (t.leaves_per_tree > 1 ? t.leaves_per_tree : 1)) return;
  if (t.depth[g] < 0) return;
  const rz_geom q = rz_geom_of(t.game);
  const int lane = rz_lane(), AS = t.game.action_stride;
  typename GM::board b;
  GM::load_leaf(b, t, g);
  const int n_stones = GM::stone_count(b);     // len(env.states)
  uint32_t h = 0;
  if (eval_id == RZ_EVAL_HASH) {
    for (int c = 0; c < 2; ++c) {
      uint32_t w = b.p[c];
      while (w) {
        const int col = __ffs(w) - 1;
        w &= w - 1;
        const uint32_t m1 = (uint32_t)(lane * q.W + col + 1);
        h += m1 * m1 * (3u + 4u * (uint32_t)c);
      }
    }
    h = rz_warp_sum_u32(h);
    h += 7u * (uint32_t)(b.last_move + 1);
    h *= 2654435761u;
  }
  float v = 0.0f;
  if (eval_id == RZ_EVAL_KAT) v = (float)((17 * n_stones + 31 * (b.last_move + 1)) % 13 - 6) / 8.0f;
  else if (eval_id == RZ_EVAL_HASH) v = (float)((int)((h >> 16) % 129u) - 64) / 64.0f;
  if (lane == 0) value[g] = v;
  const uint32_t lctx = GM::legal_ctx(b, q);
  int n_legal = 0;
  for (int s0 = 0; s0 < AS; s0 += 32) n_legal += __popc(__ballot_sync(RZ_FULL, GM::slot_legal(lctx, s0 + lane, q)));
  const float uni = n_legal > 0 ? __fdiv_rn(1.0f, (float)n_legal) : 0.0f;
  for (int s0 = 0; s0 < AS; s0 += 32) {
    const int s = s0 + lane;
    const bool legal = GM::slot_legal(lctx, s, q);
    float p = 0.0f;
    if (legal) p = (eval_id == RZ_EVAL_HASH) ? (float)(((uint32_t)s * 29u + (h >> 8)) % 32u + 1u) / 256.0f : uni;
    prior[(size_t)g * AS + s] = p;
  }
}

// Random-playout evaluator of the pure-MCTS opponent (rlzero/mcts/rollout_mcts.py):
//   priors  uniform over the legal moves                      policy_value_fn :102-108
//   value   play uniformly random legal moves to the end      _evaluate :49-74, rollout_policy :96-100
// The reference compares the winner with current_player() AFTER the playout; the env flips the
// player after every move (gomoku_env.py:67-68), so a decisive playout is worth -1 and a tie 0.
// That rule is evaluated literally here.  mode 0: r-th empty square, r uniform from a
// counter-based RNG keyed by (seed, global game id, root visit count, ply); mode 1 / 2: lowest /
// highest legal move (deterministic, for bit-exact parity tests of everything but the RNG).
__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_eval_rollout_kernel(rz_tree_desc t, int mode, unsigned long long seed, int n_limit, float* prior,
                       float* value) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  if (t.depth[g] < 0) return;
  const rz_geom q = rz_geom_of(t.game);
  const int lane = rz_lane(), H = t.game.board_size, AS = t.game.action_stride;
  rz_wboard b;
  rz_board_load(b, t.leaf_rows + (size_t)g * 2 * H, t.leaf_meta + (size_t)g * RZ_META_STRIDE, H);
  // uniform priors over the leaf's legal moves
  {
    int n_legal = 0;
    for (int s0 = 0; s0 < AS; s0 += 32) n_legal += __popc(__ballot_sync(RZ_FULL, rz_board_slot_legal(b, s0 + lane, q)));
    const float uni = n_legal > 0 ? __fdiv_rn(1.0f, (float)n_legal) : 0.0f;
    for (int s0 = 0; s0 < AS; s0 += 32) {
      const int s = s0 + lane;
      prior[(size_t)g * AS + s] = rz_board_slot_legal(b, s, q) ? uni : 0.0f;
    }
  }
  const uint32_t rowmask = (q.W >= 32) ? 0xffffffffu : ((1u << q.W) - 1u);
  const uint32_t visit = (uint32_t)t.root_N[g];
  // the stream also depends on the root position (stones on the board) and on the host's search counter
  // (rz_tree_desc.seed_dev), so that playout #v of different moves / games does not repeat the same numbers
  const uint32_t c3 = 0x7011u + ((uint32_t)t.root_meta[(size_t)g * RZ_META_STRIDE + RZ_META_STONES] << 16);
  if (t.seed_dev) seed += *t.seed_dev;
  int winner = -1;
  for (int i = 0; i < n_limit; ++i) {
    const int status = rz_board_status(b, q, winner);
    if (status != RZ_ACTIVE) break;
    // candidate squares: every empty square, or (gravity) the empty squares of the top row = open columns
    const uint32_t empty = (q.gravity ? lane == H - 1 : lane < H) ? (~(b.p[0] | b.p[1]) & rowmask) : 0u;
    const int cnt = __popc(empty);
    int inc = cnt;  // inclusive prefix count of empty squares over the rows
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(RZ_FULL, inc, o);
      if (lane >= o) inc += up;
    }
    const int n_legal = __shfl_sync(RZ_FULL, inc, 31);
    int r;
    if (mode == 1) r = 0;
    else if (mode == 2) r = n_legal - 1;
    else {
      uint32_t rnd[4];
      rz_philox4((uint32_t)(t.global_offset + g), visit, (uint32_t)i, c3, seed, rnd);
      r = (int)(((unsigned long long)rnd[0] * (unsigned long long)n_legal) >> 32);
    }
    // the row holding the r-th empty square, then its column
    const bool mine = (r >= inc - cnt) && (r < inc);
    const unsigned who = __ballot_sync(RZ_FULL, mine);
    const int row = __ffs(who) - 1;
    int col = 0;
    if (mine) {
      uint32_t m = empty;
      for (int j = r - (inc - cnt); j > 0; --j) m &= m - 1;
      col = __ffs(m) - 1;
    }
    col = __shfl_sync(RZ_FULL, col, row);
    rz_board_play(b, q.gravity ? col : row * q.W + col, q);
  }
  if (lane == 0) value[g] = (winner == -1) ? 0.0f : (winner == b.player ? 1.0f : -1.0f);
}

// RandomRolloutEvaluator of the DeepMindMCTS driver (rlzero/mcts/deepmind_mcts.py:31-62):
//   prior     1/len(legal) for every legal action                                  :58-62
//   evaluate  mean over n_rollouts uniformly random playouts of env.returns()       :43-56
// returns follow enum rz_returns (the reference's GomokuEnv.returns quirk included).  A playout that
// is cut by n_limit before the game ends contributes [0,0].  Counter-based RNG keyed by (seed,
// global game id, root visit count, rollout, ply).
template <class GM>
__global__ void __launch_bounds__(RZ_GAME_THREADS)
rz_eval_rollout_dm_kernel(rz_tree_desc t, int n_rollouts, unsigned long long seed, int n_limit, float* prior,
                          double* ret64) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  const int g = blockIdx.x * RZ_GAME_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  if (t.depth[g] < 0) return;
  const rz_geom q = rz_geom_of(t.game);
  const int lane = rz_lane(), AS = t.game.action_stride;
  typename GM::board b0;
  GM::load_leaf(b0, t, g);
  {
    const uint32_t lctx = GM::legal_ctx(b0, q);
    int n_legal = 0;
    for (int s0 = 0; s0 < AS; s0 += 32) n_legal += __popc(__ballot_sync(RZ_FULL, GM::slot_legal(lctx, s0 + lane, q)));
    const float uni = n_legal > 0 ? __fdiv_rn(1.0f, (float)n_legal) : 0.0f;
    for (int s0 = 0; s0 < AS; s0 += 32) {
      const int s = s0 + lane;
      prior[(size_t)g * AS + s] = GM::slot_legal(lctx, s, q) ? uni : 0.0f;
    }
  }
  const uint32_t visit = (uint32_t)t.root_N[g];
  if (t.seed_dev) seed += *t.seed_dev;   // the host's search counter (rz_tree_desc.seed_dev)
  int sum0 = 0, sum1 = 0;
  for (int r = 0; r < n_rollouts; ++r) {
    typename GM::board b = b0;
    int winner = -1, status = RZ_ACTIVE;
    for (int i = 0; i <= n_limit; ++i) {
      status = GM::status(b, q, winner);
      if (status != RZ_ACTIVE || i == n_limit) break;
      const uint32_t cand = GM::move_candidates(b, q);
      const int cnt = __popc(cand);
      int inc = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(RZ_FULL, inc, o);
        if (lane >= o) inc += up;
      }
      const int n_sq = __shfl_sync(RZ_FULL, inc, 31);
      const int n_act = n_sq + (GM::kHasPass ? 1 : 0);
      uint32_t rnd[4];
      rz_philox4((uint32_t)(t.global_offset + g), visit, ((uint32_t)r << 16) | (uint32_t)i, 0xd311u, seed, rnd);
      const int pick = (int)(((unsigned long long)rnd[0] * (unsigned long long)n_act) >> 32);
      int action;
      if (pick >= n_sq) {
        action = q.cells;                       // the pass
      } else {
        const bool mine = (pick >= inc - cnt) && (pick < inc);
        const unsigned who = __ballot_sync(RZ_FULL, mine);
        const int row = __ffs(who) - 1;
        int col = 0;
        if (mine) {
          uint32_t m = cand;
          for (int j = pick - (inc - cnt); j > 0; --j) m &= m - 1;
          col = __ffs(m) - 1;
        }
        col = __shfl_sync(RZ_FULL, col, row);
        action = GM::candidate_action(row, col, q);
      }
      GM::play(b, action, q);
    }
    int r0, r1;
    rz_game_returns(t.game.game_type, t.returns_mode, status, winner, r0, r1);
    sum0 += r0; sum1 += r1;
  }
  if (lane == 0) {
    ret64[2 * g] = (double)sum0 / (double)n_rollouts;
    ret64[2 * g + 1] = (double)sum1 / (double)n_rollouts;
  }
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
static int rz_check_line_game(const rz_game_desc* g) {
  if (rz_check_game(g)) return -1;
  RZ_REQUIRE(g->game_type != RZ_GAME_GO, "this entry point serves Gomoku / Connect Four; use the rz_go_* calls for Go");
  return 0;
}
static inline dim3 rz_grid(int n, int warps) { return dim3((unsigned)((n + warps - 1) / warps)); }

extern "C" int rz_gomoku_reset(const rz_game_desc* g, uint32_t* rows, int32_t* meta, int n_games,
                               int only_ended, void* stream) {
  if (rz_check_line_game(g)) return -1;
  RZ_REQUIRE(rows && meta && n_games >= 0, "rz_gomoku_reset: bad arguments");
  if (n_games == 0) return 0;
  rz_gomoku_reset_kernel<<<rz_grid(n_games, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream>>>(
      *g, rows, meta, n_games, only_ended);
  RZ_LAUNCH_CHECK("rz_gomoku_reset");
  return 0;
}

extern "C" int rz_gomoku_step(const rz_game_desc* g, uint32_t* rows, int32_t* meta,
                              const int32_t* actions, int32_t* reward, int32_t* win, int n_games,
                              void* stream) {
  if (rz_check_line_game(g)) return -1;
  RZ_REQUIRE(rows && meta && actions && n_games >= 0, "rz_gomoku_step: bad arguments");
  if (n_games == 0) return 0;
  rz_gomoku_step_kernel<<<rz_grid(n_games, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream>>>(
      *g, rows, meta, actions, reward, win, n_games);
  RZ_LAUNCH_CHECK("rz_gomoku_step");
  return 0;
}

extern "C" int rz_gomoku_legal_mask(const rz_game_desc* g, const uint32_t* rows, uint8_t* mask,
                                    int n_games, void* stream) {
  if (rz_check_line_game(g)) return -1;
  RZ_REQUIRE(rows && mask && n_games >= 0, "rz_gomoku_legal_mask: bad arguments");
  if (n_games == 0) return 0;
  rz_gomoku_legal_kernel<<<rz_grid(n_games, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream>>>(
      *g, rows, mask, n_games);
  RZ_LAUNCH_CHECK("rz_gomoku_legal_mask");
  return 0;
}

extern "C" int rz_gomoku_winner(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta,
                                int32_t* end, int32_t* winner, int n_games, void* stream) {
  if (rz_check_line_game(g)) return -1;
  RZ_REQUIRE(rows && meta && end && winner && n_games >= 0, "rz_gomoku_winner: bad arguments");
  if (n_games == 0) return 0;
  rz_gomoku_winner_kernel<<<rz_grid(n_games, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream>>>(
      *g, rows, meta, end, winner, n_games);
  RZ_LAUNCH_CHECK("rz_gomoku_winner");
  return 0;
}

extern "C" int rz_gomoku_encode_f32(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta,
                                    float* planes, int n_games, void* stream) {
  if (rz_check_line_game(g)) return -1;
  RZ_REQUIRE(rows && meta && planes && n_games >= 0, "rz_gomoku_encode_f32: bad arguments");
  if (n_games == 0) return 0;
  rz_gomoku_encode_f32_kernel<<<rz_grid(n_games, RZ_GAME_WARPS), RZ_GAME_THREADS, 0,
                                (cudaStream_t)stream>>>(*g, rows, meta, planes, n_games);
  RZ_LAUNCH_CHECK("rz_gomoku_encode_f32");
  return 0;
}

extern "C" int rz_gomoku_encode_nhwc_f32(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta,
                                         float* planes, int n_games, void* stream) {
  if (rz_check_line_game(g)) return -1;
  RZ_REQUIRE(rows && meta && planes && n_games >= 0, "rz_gomoku_encode_nhwc_f32: bad arguments");
  if (n_games == 0) return 0;
  rz_gomoku_encode_nhwc_kernel<<<rz_grid(n_games, RZ_GAME_WARPS), RZ_GAME_THREADS, 0,
                                 (cudaStream_t)stream>>>(*g, rows, meta, planes, n_games);
  RZ_LAUNCH_CHECK("rz_gomoku_encode_nhwc_f32");
  return 0;
}

extern "C" int rz_eval_rollout(const rz_tree_desc* t, int mode, unsigned long long seed, int n_limit,
                               float* prior, float* value, void* stream) {
  RZ_REQUIRE(t && prior && value, "rz_eval_rollout: null argument");
  if (rz_check_game(&t->game)) return -1;
  RZ_REQUIRE(mode >= 0 && mode <= 2, "rz_eval_rollout: mode %d", mode);
  RZ_REQUIRE(n_limit >= 0, "rz_eval_rollout: n_limit %d", n_limit);
  RZ_REQUIRE(t->root_N && t->depth && t->leaf_rows && t->leaf_meta, "rz_eval_rollout: null tree array");
  RZ_REQUIRE(t->game.game_type != RZ_GAME_GO, "rz_eval_rollout: not implemented for Go");
  RZ_REQUIRE(t->leaves_per_tree <= 1, "rz_eval_rollout: leaf-parallel waves are not supported by the rollout evaluator");
  if (t->n_trees == 0) return 0;
  rz_launch_pdl(rz_eval_rollout_kernel, rz_grid(t->n_trees, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream, *t, mode, seed, n_limit, prior, value);
  RZ_LAUNCH_CHECK("rz_eval_rollout");
  return 0;
}

extern "C" int rz_eval_closed_form(const rz_tree_desc* t, int eval_id, float* prior, float* value,
                                   void* stream) {
  RZ_REQUIRE(t && prior && value, "rz_eval_closed_form: null argument");
  if (rz_check_game(&t->game)) return -1;
  RZ_REQUIRE(eval_id >= RZ_EVAL_ZERO && eval_id <= RZ_EVAL_HASH, "rz_eval_closed_form: eval_id %d", eval_id);
  if (t->n_trees == 0) return 0;
  const int n_leaves = t->n_trees * (t->leaves_per_tree > 1 ? t->leaves_per_tree : 1);
  if (t->game.game_type == RZ_GAME_GO)
    rz_launch_pdl(rz_eval_closed_form_kernel<rz_go_game>, rz_grid(n_leaves, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream, *t, eval_id, prior, value);
  else
    rz_launch_pdl(rz_eval_closed_form_kernel<rz_line_game>, rz_grid(n_leaves, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream, *t, eval_id, prior, value);
  RZ_LAUNCH_CHECK("rz_eval_closed_form");
  return 0;
}

extern "C" int rz_eval_rollout_dm(const rz_tree_desc* t, int n_rollouts, unsigned long long seed, int n_limit,
                                  float* prior, double* ret64, void* stream) {
  RZ_REQUIRE(t && prior && ret64, "rz_eval_rollout_dm: null argument");
  if (rz_check_game(&t->game)) return -1;
  RZ_REQUIRE(n_rollouts >= 1, "rz_eval_rollout_dm: n_rollouts %d", n_rollouts);
  RZ_REQUIRE(n_limit >= 0, "rz_eval_rollout_dm: n_limit %d", n_limit);
  RZ_REQUIRE(t->root_N && t->depth && t->leaf_rows && t->leaf_meta, "rz_eval_rollout_dm: null tree array");
  RZ_REQUIRE(t->game.game_type != RZ_GAME_GO || t->leaf_hist, "rz_eval_rollout_dm: Go needs leaf_hist");
  RZ_REQUIRE(t->leaves_per_tree <= 1, "rz_eval_rollout_dm: leaf-parallel waves are not supported by the rollout evaluator");
  if (t->n_trees == 0) return 0;
  if (t->game.game_type == RZ_GAME_GO)
    rz_launch_pdl(rz_eval_rollout_dm_kernel<rz_go_game>, rz_grid(t->n_trees, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream, *t, n_rollouts, seed, n_limit, prior, ret64);
  else
    rz_launch_pdl(rz_eval_rollout_dm_kernel<rz_line_game>, rz_grid(t->n_trees, RZ_GAME_WARPS), RZ_GAME_THREADS, 0, (cudaStream_t)stream, *t, n_rollouts, seed, n_limit, prior, ret64);
  RZ_LAUNCH_CHECK("rz_eval_rollout_dm");
  return 0;
}
