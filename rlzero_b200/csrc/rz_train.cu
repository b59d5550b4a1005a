// rlzero_b200 -- training-side data kernels that consume the self-play trajectory records
// without leaving HBM (SURVEY.md 8 f1).
//
// Reference: TrainPipeline.get_equi_data (tools/train_alphazero.py:59-79): every recorded ply
// (state planes [4][H][W], pi [H*W], z) is expanded into its 8 board symmetries, in this order:
//   for i in 1..4:  rot90(state, i), then fliplr of that
// The policy vector goes through flipud o rot90^i o flipud (and fliplr in between for the flipped
// copies) -- literally what the reference does, including the fact that this is NOT the same
// geometric map as the one applied to the planes (the reference kept upstream's flipud although
// its current_state is not flipped).  Parity is bit-for-bit data movement: no arithmetic.
#include "rz_common.cuh"

namespace {

// source coordinates of rot90 applied `i` times: out[r][c] = in[R1^i(r, c)], R1(r, c) = (c, N-1-r)
__device__ __forceinline__ void rot_src(int i, int N, int& r, int& c) {
  for (int t = 0; t < i; ++t) {
    const int nr = c, nc = N - 1 - r;
    r = nr; c = nc;
  }
}

__global__ void __launch_bounds__(256)
rz_augment_equi_kernel(rz_game_desc gd, const uint32_t* __restrict__ rows, const int32_t* __restrict__ info,
                       int info_stride, const float* __restrict__ pi, float* __restrict__ out_planes,
                       float* __restrict__ out_pi, float* __restrict__ out_z, int n) {
  const int H = gd.board_size, A = gd.n_actions, AS = gd.action_stride;
  const long long total = (long long)n * 8 * A;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int cell = (int)(idx % A);
    const long long rec8 = idx / A;
    const int sym = (int)(rec8 & 7);          // 2*(i-1) + flipped
    const int rec = (int)(rec8 >> 3);
    const int i = (sym >> 1) + 1, flipped = sym & 1;
    const int r = cell / H, c = cell - r * H;
    // planes: out[r][c] = state[R1^i(r, flipped ? N-1-c : c)]
    int sr = r, sc = flipped ? H - 1 - c : c;
    rot_src(i, H, sr, sc);
    const int32_t* inf = info + (size_t)rec * info_stride;
    const int mover = inf[0], last = inf[1];
    const uint32_t* rw = rows + (size_t)rec * 2 * H;
    const uint32_t mine = rw[mover * H + sr], theirs = rw[(mover ^ 1) * H + sr];
    int stones = 0;
    for (int y = 0; y < H; ++y) stones += __popc(rw[y]) + __popc(rw[H + y]);
    float* op = out_planes + ((size_t)rec8 * 4) * A + cell;
    op[0] = (float)((mine >> sc) & 1u);                                   // gomoku_env.py:100-106
    op[A] = (float)((theirs >> sc) & 1u);
    op[2 * A] = (stones > 0 && last == sr * H + sc) ? 1.0f : 0.0f;        // :108
    op[3 * A] = (stones & 1) ? 0.0f : 1.0f;                               // :110-111
    // pi: out[r][c] = P[N-1-a][b], (a, b) = R1^i(N-1-r, flipped ? N-1-c : c)
    int a = H - 1 - r, b = flipped ? H - 1 - c : c;
    rot_src(i, H, a, b);
    out_pi[(size_t)rec8 * A + cell] = pi[(size_t)rec * AS + (H - 1 - a) * H + b];
    if (cell == 0) out_z[rec8] = (float)inf[2];
  }
}

// gather rows of a [cap][width] float table: dst[i] = src[index[i]]  (replay-buffer mini-batches)
__global__ void __launch_bounds__(256)
rz_gather_rows_kernel(const float* __restrict__ src, const long long* __restrict__ index, float* __restrict__ dst,
                      int n, int width) {
  const long long total = (long long)n * width;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(idx / width), col = (int)(idx - (long long)row * width);
    dst[idx] = src[index[row] * width + col];
  }
}

// ---- Go training records -------------------------------------------------------------------------------------------
// A Go position's 17 GoEnv.observe planes (go_env.py:156-178) are eight (position, colour) pairs plus the mover.  The
// ring stores only the board of each ply, so the history is rebuilt here from the preceding records of the same episode,
// which the ring holds consecutively, and kept as row bitmasks: 16 x H words per record instead of 8 augmented float
// copies of 17 x H x W planes.  The symmetries are applied when a mini-batch is expanded.
#define RZ_GO_REC_WARPS 8

// One warp per written record, lane = board row.  Entry e of record i comes from src = i - e when src has the same slot
// (info[3]), the same episode (info[4]), ply[src] == ply[i] - e and ply[src] >= 1: plane 2e = the stones of src's
// previous mover, plane 2e + 1 = the stones of src's mover; zero otherwise (BatchedSelfPlay._go_states).  Every input
// record serves as history; only the newest `capacity` are written, record i to slot (dst_start + i) % capacity.
__global__ void __launch_bounds__(RZ_GO_REC_WARPS * 32)
rz_go_records_pack_kernel(int H, int A, int AS, const uint32_t* __restrict__ rows, const int32_t* __restrict__ info,
                          int info_stride, const float* __restrict__ pi, int n, int first, uint32_t* __restrict__ planes,
                          int32_t* __restrict__ mover_out, float* __restrict__ pi_out, float* __restrict__ z_out,
                          int capacity, int dst_start) {
  const int i = first + blockIdx.x * RZ_GO_REC_WARPS + (threadIdx.x >> 5);
  if (i >= n) return;
  const int lane = rz_lane();
  const int32_t* inf = info + (size_t)i * info_stride;
  const int slot = inf[3], episode = inf[4], ply = inf[5];
  const size_t dst = (size_t)(((long long)dst_start + i) % capacity);
  uint32_t* op = planes + dst * 16 * H;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int src = i - e;
    uint32_t prev = 0u, cur = 0u;
    if (src >= 0) {
      const int32_t* si = info + (size_t)src * info_stride;
      if (si[3] == slot && si[4] == episode && si[5] == ply - e && si[5] >= 1 && lane < H) {
        const int m = si[0];
        const uint32_t* rw = rows + (size_t)src * 2 * H;
        prev = rw[(1 - m) * H + lane];
        cur = rw[m * H + lane];
      }
    }
    if (lane < H) {
      op[(2 * e) * H + lane] = prev;
      op[(2 * e + 1) * H + lane] = cur;
    }
  }
  const float* ps = pi + (size_t)i * AS;
  float* pd = pi_out + dst * A;
  for (int a = lane; a < A; a += 32) pd[a] = ps[a];
  if (lane == 0) {
    mover_out[dst] = inf[0];
    z_out[dst] = (float)inf[2];
  }
}

// One block per (slot, symmetry) pair -> the 17 planes [17][H][W], pi [A] and z of AlphaZeroAgent.learn.  Symmetry s is
// one of rz_augment_equi's 8 plane maps, in its order: rot90 applied s / 2 + 1 times, then fliplr when s is odd (s = 6
// is the identity).  The H*W square probabilities go through the SAME map as the planes and the pass stays last: Go has
// no reference training pipeline to keep parity with, so the geometrically consistent map is the definition (unlike
// rz_augment_equi's policy map, which keeps the reference's flipud quirk).  slot and sym come from device memory, which
// the host cannot check: only slot % capacity and sym & 7 are read.
__global__ void __launch_bounds__(256)
rz_go_records_expand_kernel(int H, int A, const uint32_t* __restrict__ planes, const int32_t* __restrict__ mover,
                            const float* __restrict__ pi, const float* __restrict__ z, int capacity,
                            const long long* __restrict__ slots, const long long* __restrict__ syms, int n,
                            float* __restrict__ out_states, float* __restrict__ out_pi, float* __restrict__ out_z) {
  __shared__ uint32_t sp[16 * RZ_MAX_BOARD];
  const int b = blockIdx.x;
  long long s64 = slots[b] % capacity;
  if (s64 < 0) s64 += capacity;
  const size_t slot = (size_t)s64;
  const int sym = (int)(syms[b] & 7);
  const int i = (sym >> 1) + 1, flipped = sym & 1;
  const int HW = H * H;
  for (int t = threadIdx.x; t < 16 * H; t += blockDim.x) sp[t] = planes[slot * 16 * H + t];
  __syncthreads();
  const float m1 = mover[slot] == 1 ? 1.0f : 0.0f;
  float* os = out_states + (size_t)b * 17 * HW;
  const float* ps = pi + slot * A;
  float* opi = out_pi + (size_t)b * A;
  for (int cell = threadIdx.x; cell < HW; cell += blockDim.x) {
    const int r = cell / H, c = cell - r * H;
    int sr = r, sc = flipped ? H - 1 - c : c;        // out[r][c] = in[R1^i(r, flipped ? N-1-c : c)]
    rot_src(i, H, sr, sc);
#pragma unroll
    for (int p = 0; p < 16; ++p) os[p * HW + cell] = (float)((sp[p * H + sr] >> sc) & 1u);
    os[16 * HW + cell] = m1;
    opi[cell] = ps[sr * H + sc];
  }
  if (threadIdx.x == 0) {
    opi[A - 1] = ps[A - 1];                          // the pass
    out_z[b] = z[slot];
  }
}

}  // namespace

static int rz_check_go_records(const rz_game_desc* g, const char* who, int capacity) {
  if (rz_check_go(g, who)) return -1;
  RZ_REQUIRE(capacity >= 1, "%s: capacity %d < 1", who, capacity);
  return 0;
}

extern "C" int rz_go_records_pack(const rz_game_desc* g, const uint32_t* rows, const int32_t* info, int info_stride,
                                  const float* pi, int n, uint32_t* planes, int32_t* mover, float* out_pi, float* z,
                                  int capacity, int dst_start, void* stream) {
  if (rz_check_go_records(g, "rz_go_records_pack", capacity)) return -1;
  RZ_REQUIRE(rows, "rz_go_records_pack: rows is null");
  RZ_REQUIRE(info, "rz_go_records_pack: info is null");
  RZ_REQUIRE(pi, "rz_go_records_pack: pi is null");
  RZ_REQUIRE(planes, "rz_go_records_pack: planes is null");
  RZ_REQUIRE(mover, "rz_go_records_pack: mover is null");
  RZ_REQUIRE(out_pi, "rz_go_records_pack: out_pi is null");
  RZ_REQUIRE(z, "rz_go_records_pack: z is null");
  RZ_REQUIRE(n >= 0, "rz_go_records_pack: n %d < 0", n);
  RZ_REQUIRE(info_stride >= 6, "rz_go_records_pack: info_stride %d < 6 (mover, last_move, z, slot, episode, ply)",
             info_stride);
  RZ_REQUIRE(dst_start >= 0 && dst_start < capacity, "rz_go_records_pack: dst_start %d outside [0, capacity %d)",
             dst_start, capacity);
  const int first = n > capacity ? n - capacity : 0;
  const int n_write = n - first;
  if (n_write == 0) return 0;
  rz_go_records_pack_kernel<<<(n_write + RZ_GO_REC_WARPS - 1) / RZ_GO_REC_WARPS, RZ_GO_REC_WARPS * 32, 0,
                              (cudaStream_t)stream>>>(g->board_size, g->n_actions, g->action_stride, rows, info,
                                                      info_stride, pi, n, first, planes, mover, out_pi, z, capacity,
                                                      dst_start);
  RZ_LAUNCH_CHECK("rz_go_records_pack");
  return 0;
}

extern "C" int rz_go_records_expand(const rz_game_desc* g, const uint32_t* planes, const int32_t* mover,
                                    const float* pi, const float* z, int capacity, const long long* slots,
                                    const long long* syms, int n, float* out_states, float* out_pi, float* out_z,
                                    void* stream) {
  if (rz_check_go_records(g, "rz_go_records_expand", capacity)) return -1;
  RZ_REQUIRE(planes, "rz_go_records_expand: planes is null");
  RZ_REQUIRE(mover, "rz_go_records_expand: mover is null");
  RZ_REQUIRE(pi, "rz_go_records_expand: pi is null");
  RZ_REQUIRE(z, "rz_go_records_expand: z is null");
  RZ_REQUIRE(slots, "rz_go_records_expand: slots is null");
  RZ_REQUIRE(syms, "rz_go_records_expand: syms is null");
  RZ_REQUIRE(out_states, "rz_go_records_expand: out_states is null");
  RZ_REQUIRE(out_pi, "rz_go_records_expand: out_pi is null");
  RZ_REQUIRE(out_z, "rz_go_records_expand: out_z is null");
  RZ_REQUIRE(n >= 0, "rz_go_records_expand: n %d < 0", n);
  if (n == 0) return 0;
  rz_go_records_expand_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(g->board_size, g->n_actions, planes, mover, pi, z,
                                                                   capacity, slots, syms, n, out_states, out_pi,
                                                                   out_z);
  RZ_LAUNCH_CHECK("rz_go_records_expand");
  return 0;
}

extern "C" int rz_augment_equi(const rz_game_desc* g, const uint32_t* rows, const int32_t* info, int info_stride,
                               const float* pi, float* out_planes, float* out_pi, float* out_z, int n,
                               void* stream) {
  if (rz_check_game(g)) return -1;
  // the 4-plane Gomoku encoding with H*H actions on a square board; anything else would be read out of range
  RZ_REQUIRE(g->game_type == RZ_GAME_GOMOKU,
             "rz_augment_equi: game_type %d: only square Gomoku boards (Go records: rz_go_records_pack / "
             "rz_go_records_expand)", g->game_type);
  RZ_REQUIRE(g->width <= 0 || g->width == g->board_size,
             "rz_augment_equi: width %d != board_size %d: only square Gomoku boards", g->width, g->board_size);
  RZ_REQUIRE(rows && info && pi && out_planes && out_pi && out_z, "rz_augment_equi: null argument");
  RZ_REQUIRE(info_stride >= 3 && n >= 0, "rz_augment_equi: bad sizes");
  if (n == 0) return 0;
  const long long total = (long long)n * 8 * g->n_actions;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  rz_augment_equi_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(*g, rows, info, info_stride, pi, out_planes,
                                                                  out_pi, out_z, n);
  RZ_LAUNCH_CHECK("rz_augment_equi");
  return 0;
}

extern "C" int rz_gather_rows(const float* src, const long long* index, float* dst, int n, int width,
                              void* stream) {
  RZ_REQUIRE(src && index && dst && n >= 0 && width >= 1, "rz_gather_rows: bad arguments");
  if (n == 0) return 0;
  const long long total = (long long)n * width;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  rz_gather_rows_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(src, index, dst, n, width);
  RZ_LAUNCH_CHECK("rz_gather_rows");
  return 0;
}
