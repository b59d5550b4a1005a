// rlzero_b200 -- the batched 15x15 trunk behind the stem in ONE launch: each CTA pair carries chunks of its boards
// through every layer, the activations between layers kept in an L2-sized scratch.
//
// Reference op: the 3x3 convolution stack of the ResNet-N policy-value trunk (SURVEY.md section 7) between the stem and
// the heads, + the heads' two 1x1 convolutions (policy_value_net.py:41,47), for the thousands of leaves a search wave
// evaluates at once.
//
// Why: the per-layer path (rz_net_tc2.cu) launches once per layer, and every layer reads its input from HBM and writes
// its output back (every second one also reads the skip input): 537 MB per tensor at 8192 boards, ~26 GB per ResNet-10
// wave.  Under the board power limit those bytes cost clock: the same 20 launches with all tiles confined to a 16 MB
// window of L2 run 11 % faster at 1519 against 1375 MHz (profiles/r3_step0_conv_l2_probe.log, B200 at 1000 W).  Here
//   * pair p owns a contiguous range of boards and walks it in chunks of at most `chunk` boards; for each chunk it runs
//     layer after layer over the chunk's boards (one board = one 256-row pair tile, exactly tc2's tile and MMA
//     sequence, so every board gets the bits the per-layer path gives it);
//   * a layer's output goes to a per-pair scratch of two tensors T / X of chunk x 256 rows (0.75 MB per pair at chunk 6,
//     55 MB for 74 pairs: it stays in the 126 MB L2; DESIGN §3.8 has the measured chunk sweep).  Layer l writes buffer l & 1 and reads buffer (l-1) & 1 (layer 0:
//     the stem's output); a skip input, the activation two layers back, is buffer l & 1 itself (layer 1: the stem's
//     output), so the epilogue reads its residual row and then overwrites it in place;
//   * hand-over: the epilogue stores with generic stores, fence.proxy.async, and arrives on the slot's cluster-scope
//     "stored" barrier in both CTAs; the producer waits on it before it loads the slot's tile for the next layer;
//   * the 9 weight taps of a layer stay resident (147 KB per CTA, as in tc2).  At a layer boundary tap t of the next
//     layer is reloaded as soon as the previous layer's last tile has issued its tap-t MMAs (a per-tap "free"
//     tcgen05.commit), so the reload lands behind the remaining taps' MMAs;
//   * the last layer applies the heads' 1x1 convolutions in its epilogue and writes only the 6 features per square,
//     as rz_conv3x3_tc2_kernel<true> does.
// Halo rows: a tile reads 17 rows of the neighbouring slots.  Those above a board are its neighbour's pad rows, which
// every epilogue writes as zero (and the scratch starts zeroed), so they are zero as in the per-layer path; those below
// it feed only pad outputs, which the epilogue zeroes with a select, so stale values there are harmless.
#include <cuda_bf16.h>

#include "rz_common.cuh"
#include "rz_tc.cuh"

namespace {

constexpr int TILE_M = 128;
constexpr int HALO = 17;                          // |16*dy + dx| <= 17
constexpr int A_ROWS = TILE_M + 2 * HALO;         // 162
constexpr int A_KB_BYTES = A_ROWS * 128;          // one k-block (64 channels) of the halo tile
constexpr int A_BUF_BYTES = 2 * A_KB_BYTES;       // 41472
constexpr int B_TILE_BYTES = 64 * 128;            // 64 output channels x 64 input channels
constexpr int B_BYTES = 9 * 2 * B_TILE_BYTES;     // 147456
constexpr int CTRL_OFF = B_BYTES + 2 * A_BUF_BYTES;  // 230400
constexpr int SMEM_BYTES = CTRL_OFF + 1024;       // 231424 <= 232448
constexpr int NUM_THREADS = 320;                  // producer warp, MMA warp, 8 epilogue warps
constexpr int MAX_LAYERS = 24;
constexpr int MAX_CHUNK = 16;
constexpr int ACC_N = 128;

struct TrunkTc2Params {
  const __nv_bfloat16* act_in;     // [n_boards * 256][128]: the stem's output
  __nv_bfloat16* scratch;          // [2][n_pairs][chunk][256][128]
  int n_layers;
  unsigned relu_mask, res_mask;    // bit l: ReLU after layer l / layer l adds the activation two layers back
  int chunk;                       // boards per chunk (at most)
  int n_boards;
  int board, board_w;
};

// the launch parameters also carry the biases of every layer: the epilogue reads them from the constant bank
struct HeadTapsT {
  float w[6 * 128];                // [filter][channel]
  float b[6];
  float bias[MAX_LAYERS * 128];    // [layer][channel]
  float* feat;                     // [n_boards][6][256] float32, position index p = y*16 + x
};

// the tiles a pair runs, in order: chunk by chunk, layer by layer, board by board.  Pair `pair` of `n_pairs` owns
// boards [first, first + count), as balanced as the per-layer kernel's round robin; its chunks are balanced too, so none
// is smaller than about half of `chunk`.
struct TileSeq {
  int first, count, n_chunks;      // the pair's boards and chunks
  int c, coff, sz;                 // current chunk, its first board (relative to `first`), its size
  int l, j;                        // layer, slot (board within the chunk)
  __device__ void init(int pair, int n_pairs, int n_boards, int chunk) {
    const int base = n_boards / n_pairs, rem = n_boards % n_pairs;
    first = pair * base + min(pair, rem);
    count = base + (pair < rem ? 1 : 0);
    n_chunks = (count + chunk - 1) / chunk;
    c = 0; coff = 0; l = 0; j = 0;
    sz = chunk_size(0);
  }
  __device__ int chunk_size(int cc) const {
    return n_chunks ? count / n_chunks + (cc < count % n_chunks ? 1 : 0) : 0;
  }
  __device__ bool done() const { return c >= n_chunks; }
  __device__ int board() const { return first + coff + j; }
  __device__ void next(int n_layers) {
    if (++j < sz) return;
    j = 0;
    if (++l < n_layers) return;
    l = 0;
    coff += sz;
    sz = chunk_size(++c);
  }
};

__device__ __forceinline__ void mbar_wait_acq_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

__global__ void __launch_bounds__(NUM_THREADS, 1)
rz_conv3x3_trunk_kernel(const __grid_constant__ CUtensorMap tmap_act, const __grid_constant__ CUtensorMap tmap_scr,
                        const __grid_constant__ CUtensorMap tmap_w, const TrunkTc2Params p,
                        const __grid_constant__ HeadTapsT head) {
  // 2 accumulators of 128 columns + two 8-column slots for the fused heads' hand-over (power of two)
  constexpr int TMEM_COLS = 512;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = rz::smem_u32(smem_raw);
  const uint32_t a_base = smem_base + B_BYTES;
  const uint32_t ctrl = smem_base + CTRL_OFF;
  uint8_t* ctrl_ptr = smem_raw + CTRL_OFF;
  const uint32_t bar_afull = ctrl + 8, bar_aempty = ctrl + 24, bar_tfull = ctrl + 40, bar_tempty = ctrl + 56;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ctrl_ptr + 72);
  // per tap: weights landed (leader, both CTAs' bytes) / the previous layer's last tile is done with them (both CTAs)
  const uint32_t bar_wfull = ctrl + 128, bar_wfree = ctrl + 200;
  // per chunk slot: the slot's rows of the last layer are stored by both CTAs' epilogues (both CTAs, 16 arrivals)
  const uint32_t bar_stored = ctrl + 272;

  const int warp = rz::uniform_i32((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const uint32_t rank = rz::uniform_u32(rz::cluster_ctarank());
  const int half = (int)rank;
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int L = p.n_layers;

  if (threadIdx.x == 0 && (smem_base & 1023u)) __trap();  // layout below assumes a 1024-byte base
  if (warp == 0 && lane == 0) {
    rz::tma_prefetch_desc(&tmap_act);
    rz::tma_prefetch_desc(&tmap_scr);
    rz::tma_prefetch_desc(&tmap_w);
    for (int tap = 0; tap < 9; ++tap) { rz::mbar_init(bar_wfull + 8 * tap, 1); rz::mbar_init(bar_wfree + 8 * tap, 1); }
    for (int b = 0; b < 2; ++b) {
      rz::mbar_init(bar_afull + 8 * b, 1);
      rz::mbar_init(bar_aempty + 8 * b, 1);
      rz::mbar_init(bar_tfull + 8 * b, 1);
      rz::mbar_init(bar_tempty + 8 * b, 16);
    }
    for (int s = 0; s < MAX_CHUNK; ++s) rz::mbar_init(bar_stored + 8 * s, 16);
    rz::fence_barrier_init();
  }
  if (warp == 1) { rz::tmem_alloc_pair(rz::smem_u32(tmem_holder), TMEM_COLS); rz::tmem_relinquish_pair(); }
  rz::tc_fence_before();
  rz::cluster_sync_all();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // first scratch row of slot j in buffer b (T = 0, X = 1) of this pair
  auto scr_row = [&](int b, int j) -> int { return ((b * n_pairs + pair) * p.chunk + j) * 256; };

  // the weights are static (packed and synchronised before any forward): thread 0 requests layer 0's before the grid
  // dependency resolves, everything else waits for the stem first
  if (threadIdx.x != 0) { rz::grid_dep_wait(); rz::grid_dep_launch(); }
  if (warp == 0) {
    // ===== TMA producer (every CTA loads its own operands; completion is credited to the leader) =====
    if (lane == 0) {
      // reload > 0: tap t waits until the previous layer's last tile has finished its tap-t MMAs
      auto load_weights = [&](int layer, int reload) {
        for (int tap = 0; tap < 9; ++tap) {
          if (reload > 0) rz::mbar_wait(bar_wfree + 8 * tap, (uint32_t)(reload - 1) & 1u);
          const uint32_t l_wfull = rz::mapa_shared(bar_wfull + 8 * tap, 0);
          if (leader) rz::mbar_expect_tx(bar_wfull + 8 * tap, (uint32_t)(2 * 2 * B_TILE_BYTES));
          for (int kb = 0; kb < 2; ++kb) {
            const uint32_t dst = smem_base + (uint32_t)(tap * 2 + kb) * B_TILE_BYTES;
            rz::tma_load_2d_pair(dst, &tmap_w, l_wfull, kb * 64, (layer * 9 + tap) * 128 + half * 64);
          }
        }
      };
      TileSeq s;
      s.init(pair, n_pairs, p.n_boards, p.chunk);
      if (!s.done()) load_weights(0, 0);
      rz::grid_dep_wait();
      rz::grid_dep_launch();
      uint32_t stored_par = 0;     // bit j: parity of the next phase of slot j's "stored" barrier
      int it = 0, wl = 0;          // tiles, weight loads so far
      for (; !s.done(); s.next(L), ++it) {
        const int buf = it & 1;
        rz::mbar_wait(bar_aempty + 8 * buf, ((uint32_t)(it >> 1) & 1u) ^ 1u);
        int row0;
        const CUtensorMap* tm;
        if (s.l == 0) {
          row0 = s.board() * 256;
          tm = &tmap_act;
        } else {
          // the slot's rows of layer l-1, written by both CTAs' epilogues (generic stores, then a proxy fence)
          mbar_wait_acq_cluster(bar_stored + 8 * s.j, (stored_par >> s.j) & 1u);
          stored_par ^= 1u << s.j;
          row0 = scr_row((s.l - 1) & 1, s.j);
          tm = &tmap_scr;
        }
        row0 += (int)rank * TILE_M - HALO;
        const uint32_t l_afull = rz::mapa_shared(bar_afull + 8 * buf, 0);
        if (leader) rz::mbar_expect_tx(bar_afull + 8 * buf, (uint32_t)(2 * 2 * A_KB_BYTES));
        for (int kb = 0; kb < 2; ++kb) {
          const uint32_t dst = a_base + (uint32_t)buf * A_BUF_BYTES + (uint32_t)kb * A_KB_BYTES;
          rz::tma_load_2d_pair(dst, tm, l_afull, kb * 64, row0);
        }
        if (s.j == 0 && it > 0) {
          // the layer's weights, tap by tap as the previous layer's last tile releases them (behind the first tile's
          // activation, which does not depend on them)
          load_weights(s.l, ++wl);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp of the leader CTA runs the loop (converged, uniform operands); one elected lane
    // issues each tcgen05.mma / commit.  Per tile exactly rz_conv3x3_tc2_kernel's sequence. =====
    if (leader) {
      const uint32_t idesc = rz::umma_idesc_bf16(256, ACC_N);
      const uint32_t issue = rz::elect_one();
      const uint32_t tmem_u = rz::uniform_u32(tmem_base);
      TileSeq s;
      s.init(pair, n_pairs, p.n_boards, p.chunk);
      int it = 0, wl = 0;
      for (; !s.done(); s.next(L), ++it) {
        const int buf = it & 1;
        const uint32_t par = (uint32_t)(it >> 1) & 1u;
        const bool first = s.j == 0;
        // the last tile of this layer releases the weights to the next layer's load (if there is one)
        const bool release = s.j == s.sz - 1 && !(s.c == s.n_chunks - 1 && s.l == L - 1);
        if (first && it > 0) ++wl;
        rz::mbar_wait(bar_tempty + 8 * buf, par ^ 1u);
        rz::mbar_wait(bar_afull + 8 * buf, par);
        rz::tc_fence_after();
        const uint32_t d_tmem = tmem_u + (uint32_t)(buf * ACC_N);
        const uint32_t a_buf = a_base + (uint32_t)buf * A_BUF_BYTES;
        uint32_t acc = 0;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
          const int shift = HALO + (tap / 3 - 1) * 16 + (tap % 3 - 1);   // 0..34 rows into the halo tile
          if (first) { rz::mbar_wait(bar_wfull + 8 * tap, (uint32_t)wl & 1u); rz::tc_fence_after(); }
          for (int kb = 0; kb < 2; ++kb) {
            const uint32_t a_addr = a_buf + (uint32_t)kb * A_KB_BYTES + (uint32_t)shift * 128u;
            const uint32_t b_addr = smem_base + (uint32_t)(tap * 2 + kb) * B_TILE_BYTES;
            const uint64_t adesc = rz::umma_desc_sw128_bo(a_addr, 0u);
            const uint64_t bdesc = rz::umma_desc_sw128(b_addr);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              rz::umma_bf16_pair_pred(d_tmem, adesc + (uint64_t)(2 * kk), bdesc + (uint64_t)(2 * kk), idesc, acc, issue);
              acc = 1;
            }
          }
          if (release) rz::umma_commit_pair_pred(bar_wfree + 8 * tap, 3, issue);
        }
        rz::umma_commit_pair_pred(bar_tfull + 8 * buf, 3, issue);
      }
    }
  } else {
    // ===== epilogue warps 2..9: TMEM lane quarter = warp % 4, channel half = (warp - 2) / 4: one output row x 64
    // channels per thread.  The arithmetic of rz_conv3x3_tc2_kernel: + bias, + residual, ReLU, bf16, pad select; in
    // the last layer that of its fused heads (the same summation order). =====
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int col0 = hsel * 64;
    const int r_in_tile = q * 32 + lane;
    const int pos = (int)rank * TILE_M + r_in_tile;     // the same square in every tile
    const bool valid = ((pos & 15) < p.board_w) && ((pos >> 4) < p.board);
    const uint32_t bar_stored_peer = rz::mapa_shared(bar_stored, rank ^ 1u);
    // residual segment of this thread's row, double-buffered in registers: the loads for the next tile are issued
    // while this one is processed
    uint32_t res[4][8], resn[4][8];
    bool next_res = false;
    auto load_res = [&](int l_, int j_, int board_) {
      next_res = ((p.res_mask >> l_) & 1u) && valid;
      if (next_res) {
        // two layers back: the stem's output for layer 1, else this layer's own output buffer (read, then overwritten)
        const __nv_bfloat16* rrow =
            (l_ == 1 ? p.act_in + (size_t)board_ * 256 * 128 : p.scratch + (size_t)scr_row(l_ & 1, j_) * 128) +
            (size_t)pos * 128 + col0;
#pragma unroll
        for (int j = 0; j < 4; ++j) rz::ld_global_v8_stream(rrow + j * 16, resn[j]);
      }
    };
    TileSeq s;
    s.init(pair, n_pairs, p.n_boards, p.chunk);
    if (!s.done()) load_res(s.l, s.j, s.board());
    int it = 0;
    for (; !s.done(); ++it) {
      const int buf = it & 1;
      const int l = s.l, slot = s.j, board = s.board();
      const bool last = l == L - 1;
      const bool relu = (p.relu_mask >> l) & 1u;
      const bool have_res = next_res;
      if (have_res) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) res[j][e] = resn[j][e];
      }
      s.next(L);
      if (!s.done()) load_res(s.l, s.j, s.board()); else next_res = false;
      rz::mbar_wait(bar_tfull + 8 * buf, (uint32_t)(it >> 1) & 1u);
      rz::tc_fence_after();
      if (warp == 2 && lane == 0) rz::mbar_arrive(bar_aempty + 8 * buf);   // MMAs done: the A tile is dead
      uint32_t acc[2][32];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch)
        rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * ACC_N + col0 + ch * 32), acc[ch]);
      rz::tmem_ld_wait();
      // accumulator drained: the MMA issuer may overwrite it (no memory payload -> relaxed)
      rz::tc_fence_before();
      __syncwarp();
      if (lane == 0) rz::mbar_arrive_cluster_relaxed(rz::mapa_shared(bar_tempty + 8 * buf, 0));
      const float4* bias4 = reinterpret_cast<const float4*>(head.bias + l * 128 + col0);
      if (!last) {
        __nv_bfloat16* orow = p.scratch + ((size_t)scr_row(l & 1, slot) + pos) * 128 + col0;
        uint32_t pair8[8];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 b0 = bias4[ch * 8 + j * 2], b1 = bias4[ch * 8 + j * 2 + 1];
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
            uint32_t packed[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = j * 8 + e * 2;
              float v0 = __uint_as_float(acc[ch][c]) + bb[e * 2];
              float v1 = __uint_as_float(acc[ch][c + 1]) + bb[e * 2 + 1];
              if (have_res) {
                const uint32_t rw = res[ch * 2 + (j >> 1)][(j & 1) * 4 + e];
                v0 += __uint_as_float(rw << 16);
                v1 += __uint_as_float(rw & 0xffff0000u);
              }
              packed[e] = relu ? rz::pack_bf16x2_relu(v0, v1) : rz::pack_bf16x2(v0, v1);
              if (!valid) packed[e] = 0u;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) pair8[(j & 1) * 4 + e] = packed[e];
            if (j & 1) rz::st_global_v8(orow + ch * 32 + (j - 1) * 8, pair8);
          }
        }
        // the rows -> visible to the TMA (async proxy) loads of the next layer in both CTAs, then "slot stored"
        fence_proxy_async_global();
        __syncwarp();
        if (lane == 0) {
          rz::mbar_arrive_cluster(rz::mapa_shared(bar_stored + 8 * slot, rank));
          rz::mbar_arrive_cluster(bar_stored_peer + 8 * slot);
        }
      } else {
        float hacc[6];
#pragma unroll
        for (int f = 0; f < 6; ++f) hacc[f] = hsel == 0 ? head.b[f] : 0.0f;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 b0 = bias4[ch * 8 + j * 2], b1 = bias4[ch * 8 + j * 2 + 1];
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = j * 8 + e * 2;
              float v0 = __uint_as_float(acc[ch][c]) + bb[e * 2];
              float v1 = __uint_as_float(acc[ch][c + 1]) + bb[e * 2 + 1];
              if (have_res) {
                const uint32_t rw = res[ch * 2 + (j >> 1)][(j & 1) * 4 + e];
                v0 += __uint_as_float(rw << 16);
                v1 += __uint_as_float(rw & 0xffff0000u);
              }
              uint32_t pk = relu ? rz::pack_bf16x2_relu(v0, v1) : rz::pack_bf16x2(v0, v1);
              if (!valid) pk = 0u;
              const float r0 = __uint_as_float(pk << 16), r1 = __uint_as_float(pk & 0xffff0000u);
              const int cc = ch * 32 + c;
#pragma unroll
              for (int f = 0; f < 6; ++f)
                hacc[f] = fmaf(r1, head.w[f * 128 + col0 + cc + 1], fmaf(r0, head.w[f * 128 + col0 + cc], hacc[f]));
            }
          }
        }
        // partial sums of channels 64..127 -> 8 spare TMEM columns of this lane quarter (slot = tile parity), read back
        // by the partner warp of the quarter
        const uint32_t t_scr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(2 * ACC_N + buf * 8);
        if (hsel == 1) {
          uint32_t hv[8];
#pragma unroll
          for (int f = 0; f < 6; ++f) hv[f] = __float_as_uint(hacc[f]);
          hv[6] = 0u; hv[7] = 0u;
          rz::tmem_st_32x8(t_scr, hv);
          rz::tmem_st_wait();
          rz::tc_fence_before();
        }
        rz::named_bar_sync(1, 256);
        if (hsel == 0) {
          rz::tc_fence_after();
          uint32_t hv[8];
          rz::tmem_ld_32x8(t_scr, hv);
          rz::tmem_ld_wait();
          float* fo = head.feat + (size_t)board * (6 * 256) + pos;
#pragma unroll
          for (int f = 0; f < 6; ++f) fo[f * 256] = fmaxf(hacc[f] + __uint_as_float(hv[f]), 0.0f);
        }
      }
    }
  }

  rz::tc_fence_before();
  rz::cluster_sync_all();
  if (warp == 1) {
    rz::tc_fence_after();
    rz::tmem_dealloc_pair(tmem_base, TMEM_COLS);
  }
}

}  // namespace

extern "C" int rz_net_trunk_tc2(const void* act_in, const void* weights, const float* biases_host, int n_layers,
                                unsigned relu_mask, unsigned res_mask, void* scratch, int chunk, int n_boards,
                                int board_size, int board_cols, const float* w1x1_host, const float* b1x1_host,
                                float* feat, int n_ctas, void* stream) {
  RZ_REQUIRE(act_in, "rz_net_trunk_tc2: act_in is null");
  RZ_REQUIRE(weights, "rz_net_trunk_tc2: weights is null");
  RZ_REQUIRE(biases_host, "rz_net_trunk_tc2: biases_host is null");
  RZ_REQUIRE(scratch, "rz_net_trunk_tc2: scratch is null");
  RZ_REQUIRE(w1x1_host && b1x1_host, "rz_net_trunk_tc2: w1x1 / b1x1 is null");
  RZ_REQUIRE(feat, "rz_net_trunk_tc2: feat is null");
  RZ_REQUIRE(n_layers >= 1 && n_layers <= MAX_LAYERS, "rz_net_trunk_tc2: n_layers %d not in [1,%d]", n_layers, MAX_LAYERS);
  RZ_REQUIRE(!(res_mask & 1u), "rz_net_trunk_tc2: res_mask %#x: the first layer has no activation two layers back", res_mask);
  RZ_REQUIRE((res_mask >> n_layers) == 0 && (relu_mask >> n_layers) == 0,
             "rz_net_trunk_tc2: relu_mask %#x / res_mask %#x name layers past n_layers %d", relu_mask, res_mask, n_layers);
  RZ_REQUIRE(chunk >= 1 && chunk <= MAX_CHUNK, "rz_net_trunk_tc2: chunk %d not in [1,%d]", chunk, MAX_CHUNK);
  RZ_REQUIRE(n_boards >= 0, "rz_net_trunk_tc2: n_boards %d", n_boards);
  RZ_REQUIRE(board_size >= 1 && board_size <= 15, "rz_net_trunk_tc2: board_size %d not in [1,15]", board_size);
  RZ_REQUIRE(board_cols >= 1 && board_cols <= 15, "rz_net_trunk_tc2: board_cols %d not in [1,15]", board_cols);
  RZ_REQUIRE(n_ctas == 0 || n_ctas >= 2, "rz_net_trunk_tc2: n_ctas %d (0 = 148, else at least one CTA pair)", n_ctas);
  if (n_boards == 0) return 0;
  int pairs = (n_ctas > 0 ? n_ctas : 148) / 2;
  const int scratch_pairs = pairs;                    // the scratch is sized for this many pairs (include/rlzero_b200.h)
  if (pairs > n_boards) pairs = n_boards;             // every pair gets at least one board
  static HeadTapsT head;   // ~3 KB: filled per call, copied into the launch parameters
  CUtensorMap tmap_act, tmap_scr, tmap_w;
  if (rz::make_tmap_2d(&tmap_act, act_in, (uint64_t)n_boards * 256, 128, A_ROWS)) return -1;
  if (rz::make_tmap_2d(&tmap_scr, scratch, (uint64_t)2 * scratch_pairs * chunk * 256, 128, A_ROWS)) return -1;
  if (rz::make_tmap_2d(&tmap_w, weights, (uint64_t)n_layers * 9 * 128, 128, 64)) return -1;
  TrunkTc2Params p;
  p.act_in = (const __nv_bfloat16*)act_in;
  p.scratch = (__nv_bfloat16*)scratch;
  p.n_layers = n_layers;
  p.relu_mask = relu_mask;
  p.res_mask = res_mask;
  p.chunk = chunk;
  p.n_boards = n_boards;
  p.board = board_size;
  p.board_w = board_cols;
  for (int i = 0; i < 6 * 128; ++i) head.w[i] = w1x1_host[i];
  for (int i = 0; i < 6; ++i) head.b[i] = b1x1_host[i];
  head.feat = feat;
  for (int i = 0; i < n_layers * 128; ++i) head.bias[i] = biases_host[i];
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(rz_conv3x3_trunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) { rz_set_error("rz_net_trunk_tc2: smem attribute: %s", cudaGetErrorString(e)); return -2; }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * pairs));
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1 + rz_pdl_attr(&attr[1]);
  cudaError_t e = cudaLaunchKernelEx(&cfg, rz_conv3x3_trunk_kernel, tmap_act, tmap_scr, tmap_w, p, head);
  if (e != cudaSuccess) { rz_set_error("rz_net_trunk_tc2: launch failed: %s", cudaGetErrorString(e)); return -2; }
  return 0;
}
