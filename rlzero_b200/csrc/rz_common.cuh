// rlzero_b200 -- shared device/host helpers (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/rlzero_b200.h"

#define RZ_WARP 32
#define RZ_FULL 0xffffffffu

// ---- host-side error plumbing ---------------------------------------------
void rz_set_error(const char* fmt, ...);

#define RZ_REQUIRE(cond, ...)        \
  do {                               \
    if (!(cond)) {                   \
      rz_set_error(__VA_ARGS__);     \
      return -1;                     \
    }                                \
  } while (0)

#define RZ_LAUNCH_CHECK(name)                                           \
  do {                                                                  \
    cudaError_t e__ = cudaGetLastError();                               \
    if (e__ != cudaSuccess) {                                           \
      rz_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
      return -2;                                                        \
    }                                                                   \
  } while (0)

// geometry of a game as the kernels use it
struct rz_geom {
  int H, W, k, A, AS, cells, gravity, go, max_moves;
  double komi;
};
__host__ __device__ inline rz_geom rz_geom_of(const rz_game_desc& d) {
  rz_geom q;
  q.H = d.board_size;
  q.W = d.width > 0 ? d.width : d.board_size;
  q.k = d.n_in_row;
  q.A = d.n_actions;
  q.AS = d.action_stride;
  q.cells = q.H * q.W;
  q.gravity = d.game_type == RZ_GAME_CONNECT4;
  q.go = d.game_type == RZ_GAME_GO;
  q.max_moves = d.max_moves;
  q.komi = (double)d.komi;
  return q;
}

static inline int rz_check_game(const rz_game_desc* g) {
  if (!g) { rz_set_error("null game desc"); return -1; }
  if (g->board_size < 1 || g->board_size > RZ_MAX_BOARD) {
    rz_set_error("board_size %d outside [1,%d]", g->board_size, RZ_MAX_BOARD); return -1; }
  const int W = g->width > 0 ? g->width : g->board_size;
  if (W < 1 || W > RZ_MAX_BOARD) { rz_set_error("width %d outside [1,%d]", W, RZ_MAX_BOARD); return -1; }
  if (g->game_type != RZ_GAME_GOMOKU && g->game_type != RZ_GAME_CONNECT4 && g->game_type != RZ_GAME_GO) {
    rz_set_error("game_type %d", g->game_type); return -1; }
  if (g->game_type == RZ_GAME_GO) {
    if (W != g->board_size) { rz_set_error("Go needs a square board, got %dx%d", g->board_size, W); return -1; }
    if (g->n_actions != g->board_size * W + 1) {
      rz_set_error("n_actions %d: Go on %dx%d has %d actions (the pass is the last)", g->n_actions, g->board_size,
                   W, g->board_size * W + 1); return -1; }
    if (g->max_moves < 0) { rz_set_error("max_moves %d", g->max_moves); return -1; }
  } else if (g->n_actions != (g->game_type == RZ_GAME_CONNECT4 ? W : g->board_size * W)) {
    rz_set_error("n_actions %d does not match the %dx%d board of game %d", g->n_actions, g->board_size, W,
                 g->game_type); return -1; }
  if (g->action_stride < g->n_actions || (g->action_stride & 31)) {
    rz_set_error("action_stride %d must be a multiple of 32 >= n_actions", g->action_stride); return -1; }
  if (g->n_in_row < 1 || g->n_in_row > (g->board_size > W ? g->board_size : W)) {
    rz_set_error("n_in_row %d outside [1,max(H,W)]", g->n_in_row); return -1; }
  if (g->row_stride != 0 && g->row_stride != 8 && g->row_stride != 16 && g->row_stride != 20) {
    rz_set_error("row_stride %d (0 = automatic, 8, 16 or 20)", g->row_stride); return -1; }
  return 0;
}

// rz_check_game, and the descriptor must be Go (entry points that only know Go's layout)
static inline int rz_check_go(const rz_game_desc* g, const char* who) {
  if (rz_check_game(g)) return -1;
  RZ_REQUIRE(g->game_type == RZ_GAME_GO, "%s: game_type %d is not RZ_GAME_GO", who, g->game_type);
  return 0;
}

// Row stride S of the padded position layout of the tensor-core network path (a board owns S*S rows of
// [128 channels] bf16, square (y, x) at row y*S + x, squares with x >= W or y >= H hold zero): the smallest of
// 8 / 16 / 20 that leaves one zero column and one zero row, or the caller's explicit choice.  Returns 0 when
// the board does not fit.  Mirrored by rlzero_b200._lib.row_stride.
static inline int rz_row_stride(int H, int W, int requested) {
  const int m = H > W ? H : W;
  if (requested != 0) return (requested == 8 || requested == 16 || requested == 20) && m < requested ? requested : 0;
  return m <= 7 ? 8 : (m <= 15 ? 16 : (m <= 19 ? 20 : 0));
}

// ---- programmatic dependent launch ------------------------------------------
// The kernels of one wave run back to back on one stream.  A kernel launched with the programmatic-serialization
// attribute may start (barrier / TMEM set-up, loads of operands no kernel of the wave writes) while its predecessor is
// still running; rz::grid_dep_wait() blocks until every earlier grid has completed and flushed.  Every kernel launched
// this way calls grid_dep_wait() BEFORE it touches anything another kernel of the stream reads or writes and only THEN
// grid_dep_launch(): a dependent can therefore start no earlier than its predecessor's own wait has returned, so its
// set-up phase sees everything that was written two or more kernels back.  RZ_PDL=0 in the environment turns the
// attribute off (the device-side instructions are then no-ops).
bool rz_pdl_enabled();
// timing probe (rz_debug_set_probe; null in production): kernels that support it write %globaltimer stamps there
extern unsigned long long* rz_probe_buffer;
static inline int rz_pdl_attr(cudaLaunchAttribute* a) {
  a->id = cudaLaunchAttributeProgrammaticStreamSerialization;
  a->val.programmaticStreamSerializationAllowed = rz_pdl_enabled() ? 1 : 0;
  return 1;
}

// ---- device helpers --------------------------------------------------------
#ifdef __CUDACC__

// <<<grid, block, smem, stream>>> with the programmatic-serialization attribute.  The kernel must begin with
// rz::grid_dep_wait(); rz::grid_dep_launch();  Errors surface through cudaGetLastError() (RZ_LAUNCH_CHECK).
template <typename... KArgs, typename... Args>
static inline void rz_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  cfg.attrs = attr;
  cfg.numAttrs = rz_pdl_attr(&attr[0]);
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

namespace rz {
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
}  // namespace rz

__device__ __forceinline__ int rz_lane() { return threadIdx.x & 31; }

__device__ __forceinline__ unsigned rz_warp_sum_u32(unsigned v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(RZ_FULL, v, o);
  return v;
}
__device__ __forceinline__ int rz_warp_sum_i32(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(RZ_FULL, v, o);
  return v;
}
__device__ __forceinline__ double rz_warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(RZ_FULL, v, o);
  return v;
}
__device__ __forceinline__ float rz_warp_sum_f32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(RZ_FULL, v, o);
  return v;
}
__device__ __forceinline__ double rz_warp_max_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(RZ_FULL, v, o));
  return v;
}
// inclusive prefix sum over the warp
__device__ __forceinline__ double rz_warp_scan_f64(double v) {
  const int lane = rz_lane();
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    double t = __shfl_up_sync(RZ_FULL, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// Philox-4x32-10: counter-based RNG, so that a game's random stream depends only on
// (seed, global game id, episode, ply, ...) and not on which GPU or slot runs it.
struct rz_philox {
  uint32_t c[4];
  uint32_t k[2];
};
__device__ __forceinline__ void rz_philox_round(uint32_t (&c)[4], const uint32_t (&k)[2]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
  uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
  uint32_t n0 = hi1 ^ c[1] ^ k[0], n1 = lo1, n2 = hi0 ^ c[3] ^ k[1], n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__device__ __forceinline__ void rz_philox4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                           unsigned long long seed, uint32_t (&out)[4]) {
  uint32_t c[4] = {c0, c1, c2, c3};
  uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    rz_philox_round(c, k);
    k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
  }
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}
// uniform in (0,1) with 53 random bits
__device__ __forceinline__ double rz_u01_53(uint32_t a, uint32_t b) {
  unsigned long long x = (((unsigned long long)a << 32) | b) >> 11;
  return ((double)x + 0.5) * (1.0 / 9007199254740992.0);
}
__device__ __forceinline__ float rz_u01_24(uint32_t a) {
  return ((float)(a >> 8) + 0.5f) * (1.0f / 16777216.0f);
}

// env.returns() of a finished game (enum rz_returns)
__device__ __forceinline__ void rz_game_returns(int game_type, int mode, int status, int winner, int& r0, int& r1) {
  r0 = 0; r1 = 0;
  if (status != RZ_ENDED_WIN) return;
  if (game_type == RZ_GAME_GO) { r0 = winner == 0 ? 1 : -1; r1 = -r0; return; }      // go_env.py:142-143
  if (mode == RZ_RETURNS_REFERENCE) { if (winner == 1) { r0 = 1; r1 = -1; } return; }  // gomoku_env.py:216-219
  r0 = winner == 0 ? 1 : -1; r1 = -r0;
}

#endif  // __CUDACC__
