// rlzero_b200 -- batched GoEnv kernels (one warp per game).
// Reference: rlzero/games/go/go_env.py (reset 212-230, step 168-210, observe 156-166,
// legal_actions 339-340, returns 350-354) over pettingzoo's go_base; rules restated in rz_go.cuh.
#include "rz_go.cuh"

#define RZ_GO_WARPS 4
#define RZ_GO_THREADS (RZ_GO_WARPS * 32)

__global__ void __launch_bounds__(RZ_GO_THREADS)
rz_go_reset_kernel(rz_game_desc gd, uint32_t* rows, uint32_t* hist, int32_t* meta, int n, int only_ended) {
  const int g = blockIdx.x * RZ_GO_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const int lane = rz_lane(), H = gd.board_size;
  int32_t* m = meta + (size_t)g * RZ_META_STRIDE;
  const int st = m[RZ_META_STATUS];
  if (only_ended && !(st == RZ_ENDED_WIN || st == RZ_ENDED_TIE)) return;
  if (lane < H) {
    rows[(size_t)g * 2 * H + lane] = 0u;
    rows[(size_t)g * 2 * H + H + lane] = 0u;
    if (hist)
      for (int i = 0; i < RZ_GO_HIST; ++i) hist[((size_t)g * RZ_GO_HIST + i) * H + lane] = 0u;
  }
  if (lane == 0) {
    m[RZ_META_PLAYER] = 0;
    m[RZ_META_LAST_MOVE] = -1;
    m[RZ_META_STONES] = 0;
    m[RZ_META_STATUS] = RZ_ACTIVE;
    m[RZ_META_WINNER] = -1;
    m[RZ_META_PLY] = 0;
    m[RZ_META_FAULT] = 0;
    m[RZ_META_EPISODE] = only_ended ? m[RZ_META_EPISODE] + 1 : 0;
    m[RZ_META_KO] = -1;
    m[RZ_META_PASSES] = 0;
  }
}

// GoEnv.step (go_env.py:168-210): play_move, history shift, is_game_over / result.
// reward[g][2] = GoEnv.rewards after the step (black, white): 0,0 until the game ends.
__global__ void __launch_bounds__(RZ_GO_THREADS)
rz_go_step_kernel(rz_game_desc gd, uint32_t* rows, uint32_t* hist, int32_t* meta, const int32_t* actions,
                  int32_t* reward, int32_t* done, int n) {
  const int g = blockIdx.x * RZ_GO_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size;
  const int a = actions[g];
  if (a < 0) return;
  int32_t* m = meta + (size_t)g * RZ_META_STRIDE;
  rz_goboard b;
  uint32_t* hp = hist ? hist + (size_t)g * RZ_GO_HIST * H : nullptr;
  rz_go_load(b, rows + (size_t)g * 2 * H, hp, m, H);
  if (m[RZ_META_STATUS] != RZ_ACTIVE || !rz_go_action_legal(b, a, q)) {   // go_base IllegalMove / dead step
    if (lane == 0) m[RZ_META_FAULT] |= RZ_FAULT_ILLEGAL_MOVE;
    return;
  }
  rz_go_play(b, a, q);
  int winner;
  const int status = rz_go_status(b, q, winner);
  rz_go_store(b, rows + (size_t)g * 2 * H, hp, H);
  if (lane == 0) {
    rz_go_store_meta(b, m);
    m[RZ_META_STATUS] = status;
    m[RZ_META_WINNER] = winner;
    m[RZ_META_PLY] += 1;
    if (done) done[g] = status != RZ_ACTIVE;
    if (reward) {
      reward[2 * g + 0] = status == RZ_ACTIVE ? 0 : (winner == 0 ? 1 : -1);
      reward[2 * g + 1] = status == RZ_ACTIVE ? 0 : (winner == 1 ? 1 : -1);
    }
  }
}

// Position.all_legal_moves (go_env.py:193-194) as a byte mask [n][H*W + 1]; a finished game has
// only the pass (go_env.py:192)
__global__ void __launch_bounds__(RZ_GO_THREADS)
rz_go_legal_kernel(rz_game_desc gd, const uint32_t* rows, const int32_t* meta, uint8_t* mask, int n) {
  const int g = blockIdx.x * RZ_GO_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size, A = gd.n_actions;
  const int32_t* m = meta + (size_t)g * RZ_META_STRIDE;
  rz_goboard b;
  rz_go_load(b, rows + (size_t)g * 2 * H, nullptr, m, H);
  const bool over = m[RZ_META_STATUS] != RZ_ACTIVE;
  const uint32_t legal = over ? 0u : rz_go_legal_rows(b, q);
  for (int s0 = 0; s0 < A; s0 += 32) {
    const int s = s0 + lane;
    const bool ok = rz_go_slot_legal(legal, s, q);
    if (s < A) mask[(size_t)g * A + s] = ok ? 1 : 0;
  }
}

// Position.score() / result() of the current position: score[g] (float64), result[g] in {1,-1,0}
__global__ void __launch_bounds__(RZ_GO_THREADS)
rz_go_score_kernel(rz_game_desc gd, const uint32_t* rows, const int32_t* meta, double* score,
                   int32_t* result, int n) {
  const int g = blockIdx.x * RZ_GO_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int H = gd.board_size;
  rz_goboard b;
  rz_go_load(b, rows + (size_t)g * 2 * H, nullptr, meta + (size_t)g * RZ_META_STRIDE, H);
  const double s = rz_go_score(b, q);
  if (rz_lane() == 0) {
    if (score) score[g] = s;
    if (result) result[g] = s > 0.0 ? 1 : (s < 0.0 ? -1 : 0);
  }
}

// GoEnv.observe (go_env.py:156-166) as float32 [n][17][H][W] (the reference's (N,N,17) array,
// channels first): planes 0..15 = board_history, plane 16 = 1 when white is to move
__global__ void __launch_bounds__(RZ_GO_THREADS)
rz_go_encode_f32_kernel(rz_game_desc gd, const uint32_t* rows, const uint32_t* hist, const int32_t* meta,
                        float* planes, int n) {
  const int g = blockIdx.x * RZ_GO_WARPS + (threadIdx.x >> 5);
  if (g >= n) return;
  const rz_geom q = rz_geom_of(gd);
  const int lane = rz_lane(), H = gd.board_size, W = q.W, cells = q.cells;
  rz_goboard b;
  rz_go_load(b, rows + (size_t)g * 2 * H, hist ? hist + (size_t)g * RZ_GO_HIST * H : nullptr,
             meta + (size_t)g * RZ_META_STRIDE, H);
  float* out = planes + (size_t)g * 17 * cells;
#pragma unroll
  for (int pl = 0; pl < 16; ++pl) {
    const uint32_t mine = pl == 0 ? rz_go_theirs(b) : (pl == 1 ? rz_go_mine(b) : b.hist[pl >= 2 ? pl - 2 : 0]);
    for (int i0 = 0; i0 < cells; i0 += 32) {
      const int i = i0 + lane, ic = i < cells ? i : 0;
      const int r = ic / W, c = ic - r * W;
      const uint32_t row = __shfl_sync(RZ_FULL, mine, r);
      if (i < cells) out[pl * cells + i] = (float)((row >> c) & 1u);
    }
  }
  for (int i = lane; i < cells; i += 32) out[16 * cells + i] = (float)b.player;
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
static inline dim3 rz_go_grid(int n) { return dim3((unsigned)((n + RZ_GO_WARPS - 1) / RZ_GO_WARPS)); }

extern "C" int rz_go_reset(const rz_game_desc* g, uint32_t* rows, uint32_t* hist, int32_t* meta, int n_games,
                           int only_ended, void* stream) {
  if (rz_check_go(g, "rz_go_reset")) return -1;
  RZ_REQUIRE(rows && meta && n_games >= 0, "rz_go_reset: bad arguments");
  if (n_games == 0) return 0;
  rz_go_reset_kernel<<<rz_go_grid(n_games), RZ_GO_THREADS, 0, (cudaStream_t)stream>>>(*g, rows, hist, meta,
                                                                                      n_games, only_ended);
  RZ_LAUNCH_CHECK("rz_go_reset");
  return 0;
}

extern "C" int rz_go_step(const rz_game_desc* g, uint32_t* rows, uint32_t* hist, int32_t* meta,
                          const int32_t* actions, int32_t* reward, int32_t* done, int n_games, void* stream) {
  if (rz_check_go(g, "rz_go_step")) return -1;
  RZ_REQUIRE(rows && meta && actions && n_games >= 0, "rz_go_step: bad arguments");
  if (n_games == 0) return 0;
  rz_go_step_kernel<<<rz_go_grid(n_games), RZ_GO_THREADS, 0, (cudaStream_t)stream>>>(*g, rows, hist, meta, actions,
                                                                                     reward, done, n_games);
  RZ_LAUNCH_CHECK("rz_go_step");
  return 0;
}

extern "C" int rz_go_legal_mask(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta, uint8_t* mask,
                                int n_games, void* stream) {
  if (rz_check_go(g, "rz_go_legal_mask")) return -1;
  RZ_REQUIRE(rows && meta && mask && n_games >= 0, "rz_go_legal_mask: bad arguments");
  if (n_games == 0) return 0;
  rz_go_legal_kernel<<<rz_go_grid(n_games), RZ_GO_THREADS, 0, (cudaStream_t)stream>>>(*g, rows, meta, mask, n_games);
  RZ_LAUNCH_CHECK("rz_go_legal_mask");
  return 0;
}

extern "C" int rz_go_score(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta, double* score,
                           int32_t* result, int n_games, void* stream) {
  if (rz_check_go(g, "rz_go_score")) return -1;
  RZ_REQUIRE(rows && meta && (score || result) && n_games >= 0, "rz_go_score: bad arguments");
  if (n_games == 0) return 0;
  rz_go_score_kernel<<<rz_go_grid(n_games), RZ_GO_THREADS, 0, (cudaStream_t)stream>>>(*g, rows, meta, score, result,
                                                                                      n_games);
  RZ_LAUNCH_CHECK("rz_go_score");
  return 0;
}

extern "C" int rz_go_encode_f32(const rz_game_desc* g, const uint32_t* rows, const uint32_t* hist,
                                const int32_t* meta, float* planes, int n_games, void* stream) {
  if (rz_check_go(g, "rz_go_encode_f32")) return -1;
  RZ_REQUIRE(rows && meta && planes && n_games >= 0, "rz_go_encode_f32: bad arguments");
  if (n_games == 0) return 0;
  rz_go_encode_f32_kernel<<<rz_go_grid(n_games), RZ_GO_THREADS, 0, (cudaStream_t)stream>>>(*g, rows, hist, meta,
                                                                                           planes, n_games);
  RZ_LAUNCH_CHECK("rz_go_encode_f32");
  return 0;
}
