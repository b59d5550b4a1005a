// rlzero_b200 -- 3x3 convolution of the policy-value trunk, revision 2: weights resident in
// shared memory, activation tile loaded once with its halo, CTA pairs (tcgen05 cta_group::2).
//
// Reference op: nn.Conv2d(C, 128, kernel_size=3, padding=1) (+ folded BatchNorm, residual add,
// ReLU), trunk of rlzero/games/gomoku/policy_value_net.py:14-16,36-38 / the ResNet-N trunk of
// SURVEY.md section 7.
//
// Data layout (bf16, channels last, one 16x16 tile of positions per board):
//   act[b][p][c], p = y*16 + x; squares with x >= H or y >= H hold ZERO in every activation
//   tensor.  With row stride 16 > H the zero column x = 15 is at once the right halo of row y
//   and the left halo of row y+1, and the zero row y = 15 is the bottom halo of board b and the
//   top halo of board b+1, so the input of tap (dy,dx) for 128 consecutive output positions is
//   simply the 128 consecutive rows starting dy*16+dx further on: no im2col buffer, no boundary
//   code (rows before the tensor start are zero-filled by TMA).
//   w[tap][cout][cin] (K-major B operand), tap = kh*3 + kw.
//
// Why: revision 1 of this convolution (since removed) streamed a 128x64 activation tile AND a
// 128x64 weight tile from L2 for every (tap, k-block) -- 128 B/clk/SM, 8.5-11 GB of L2->SM traffic
// per layer against 1.07 GB algorithmic (profiles/r1_run4_*): it was L2-bandwidth bound at ~50 %
// tensor-pipe activity.  Here
//   * the 9 x 128 x 128 weights stay in shared memory for the whole launch.  295 KB do not fit one
//     SM, so two CTAs form a pair: each keeps the 64 output channels it contributes as the B
//     operand of a cta_group::2 MMA (147 KB), the pair computes 256 positions x 128 channels;
//   * the activation tile of a CTA (128 positions) is loaded ONCE per tile together with its
//     17-row halo (162 rows x 128 channels = 41 KB, double buffered); tap (dy,dx) is the same
//     tile read 16*dy+dx rows further on, i.e. only the UMMA descriptor start address moves.
// L2->SM traffic drops to 41 KB per 128x128x1152 tile (14x less); the MMA issuer never waits
// for operands inside a tile (72 back-to-back tcgen05.mma per tile).  At the start of a launch the
// first activation tile is requested before the weights, which complete on one mbarrier per tap, so
// the first tile's MMAs begin after 16 KB of weights instead of all 147 KB.
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


struct Conv2Params {
  const float* bias;               // [128]
  const __nv_bfloat16* residual;   // [rows][128] or null
  __nv_bfloat16* out;              // [rows][128]  (flags bit 6: float [rows][128] instead)
  int n_items;                     // boards
  int board;                       // H (rows)
  int board_w;                     // W (columns)
  int kblocks;                     // Cin / 64
  int relu;
  int flags;                       // bit 0: set the descriptor base-offset field for shifted A tiles
};

// kHead: the last trunk layer also applies the heads' two 1x1 convolutions + ReLU
// (policy_value_net.py:41,47: act_conv1 128->4, val_conv1 128->2) to every output row while it is
// in registers, and writes ONLY those 6 features: the trunk output never goes to HBM.  The 6x128
// filter taps ride in the kernel parameters (constant bank): 768 FFMAs with immediate-offset
// constant operands, no shared-memory or global traffic.
struct HeadTaps {
  float w[6 * 128];                // [filter][channel]
  float b[6];
  float* feat;                     // [n_boards][6][256] float32, position index p = y*16 + x
};

template <bool kHead>
__global__ void __launch_bounds__(NUM_THREADS, 1)
rz_conv3x3_tc2_kernel(const __grid_constant__ CUtensorMap tmap_act,
                      const __grid_constant__ CUtensorMap tmap_w,
                      const __grid_constant__ CUtensorMap tmap_out, const Conv2Params p,
                      const __grid_constant__ HeadTaps head) {
  constexpr int ACC_N = 128;                       // accumulator columns per buffer
  // fused-heads layer: 16 more columns (two slots of 8) carry the upper channel half's partial sums from one warp of a
  // lane quarter to the other; the allocation is a power of two
  constexpr int TMEM_COLS = kHead ? 512 : 2 * ACC_N;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = rz::smem_u32(smem_raw);
  const uint32_t a_base = smem_base + B_BYTES;
  const uint32_t ctrl = smem_base + CTRL_OFF;
  uint8_t* ctrl_ptr = smem_raw + CTRL_OFF;
  // weights: one barrier per tap (ctrl + 640 .. 711), so the first tile's MMAs of tap t start as soon as tap t has
  // landed instead of waiting for all 147 KB; the first activation tile is requested BEFORE the weights
  const uint32_t bar_btap = ctrl + 640, bar_afull = ctrl + 8, bar_aempty = ctrl + 24;
  const uint32_t bar_tfull = ctrl + 40, bar_tempty = ctrl + 56;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ctrl_ptr + 72);
  float* s_bias = reinterpret_cast<float*>(ctrl_ptr + 128);

  // warp index and cluster rank through a shuffle: values the compiler can prove warp-uniform, so the
  // role branches below are uniform and the MMA issuer's operands live in uniform registers
  const int warp = rz::uniform_i32((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const uint32_t rank = rz::uniform_u32(rz::cluster_ctarank());
  const int half = (int)rank;                      // which 64 output channels live here
  const bool leader = rank == 0;
  const int worker = blockIdx.x >> 1, n_workers = gridDim.x >> 1;

  // flags bit 9: the weights and the bias are not written by any kernel near this one on the stream (the search's
  // network forward): they are fetched BEFORE the grid dependency resolves, i.e. while the previous layer is still
  // running (rz_common.cuh, programmatic dependent launch).  Otherwise the kernel waits first.
  const bool early_w = (p.flags & 512) != 0;
  if (!early_w) rz::grid_dep_wait();
  if (threadIdx.x == 0 && (smem_base & 1023u)) __trap();  // layout below assumes a 1024-byte base
  if (warp == 0 && lane == 0) {
    rz::tma_prefetch_desc(&tmap_act);
    rz::tma_prefetch_desc(&tmap_w);
    rz::tma_prefetch_desc(&tmap_out);
    for (int tap = 0; tap < 9; ++tap) rz::mbar_init(bar_btap + 8 * tap, 1);
    for (int b = 0; b < 2; ++b) {
      rz::mbar_init(bar_afull + 8 * b, 1);
      rz::mbar_init(bar_aempty + 8 * b, 1);
      rz::mbar_init(bar_tfull + 8 * b, 1);
      rz::mbar_init(bar_tempty + 8 * b, 16);
    }
    rz::fence_barrier_init();
  }
  if (warp == 1) { rz::tmem_alloc_pair(rz::smem_u32(tmem_holder), TMEM_COLS); rz::tmem_relinquish_pair(); }
  if (threadIdx.x >= 64 && threadIdx.x < 192) s_bias[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  rz::tc_fence_before();
  rz::cluster_sync_all();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // first row of this CTA's 128 output positions for work item `item`
  auto row_of = [&](int item) -> int {
    return item * 256 + (int)rank * TILE_M;
  };

  if (early_w && threadIdx.x != 0) rz::grid_dep_wait();   // thread 0 (the producer) first requests the weights
  if (threadIdx.x != 0) rz::grid_dep_launch();
  if (warp == 0) {
    // ===== TMA producer (every CTA loads its own operands; completion is credited to the leader) =====
    if (lane == 0) {
      auto load_weights = [&]() {
        for (int tap = 0; tap < 9; ++tap) {
          const uint32_t l_btap = rz::mapa_shared(bar_btap + 8 * tap, 0);
          if (leader) rz::mbar_expect_tx(bar_btap + 8 * tap, (uint32_t)(2 * p.kblocks * B_TILE_BYTES));
          for (int kb = 0; kb < p.kblocks; ++kb) {
            const uint32_t dst = smem_base + (uint32_t)(tap * 2 + kb) * B_TILE_BYTES;
            rz::tma_load_2d_pair(dst, &tmap_w, l_btap, kb * 64, tap * 128 + half * 64);
          }
        }
      };
      if (early_w) { if (worker < p.n_items) load_weights(); rz::grid_dep_wait(); }
      rz::grid_dep_launch();
      int it = 0;
      for (int item = worker; item < p.n_items; item += n_workers, ++it) {
        const int buf = it & 1;
        rz::mbar_wait(bar_aempty + 8 * buf, ((uint32_t)(it >> 1) & 1u) ^ 1u);
        const uint32_t l_afull = rz::mapa_shared(bar_afull + 8 * buf, 0);
        if (leader) rz::mbar_expect_tx(bar_afull + 8 * buf, (uint32_t)(2 * p.kblocks * A_KB_BYTES));
        const int row0 = row_of(item) - HALO;
        for (int kb = 0; kb < p.kblocks; ++kb) {
          const uint32_t dst = a_base + (uint32_t)buf * A_BUF_BYTES + (uint32_t)kb * A_KB_BYTES;
          rz::tma_load_2d_pair(dst, &tmap_act, l_afull, kb * 64, row0);
        }
        if (it == 0 && !early_w) load_weights();      // right behind the first activation tile
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp of the leader CTA runs the loop (converged, uniform operands);
    // one elected lane issues each tcgen05.mma / commit =====
    if (leader) {
      // flags bit 8: the layer has only 64 output channels -- N = 64 MMAs (each CTA supplies the first 32 rows of its
      // weight tiles: output channels 0..31 / 32..63), accumulator columns 0..63
      const uint32_t idesc = (p.flags & 256) ? rz::umma_idesc_bf16(256, 64) : rz::umma_idesc_bf16(256, ACC_N);
      const uint32_t issue = rz::elect_one();
      const uint32_t tmem_u = rz::uniform_u32(tmem_base);
      int it = 0;
      for (int item = worker; item < p.n_items; item += n_workers, ++it) {
        const int buf = it & 1;
        const uint32_t par = (uint32_t)(it >> 1) & 1u;
        rz::mbar_wait(bar_tempty + 8 * buf, par ^ 1u);
        rz::mbar_wait(bar_afull + 8 * buf, par);
        rz::tc_fence_after();
        const uint32_t d_tmem = tmem_u + (uint32_t)(buf * ACC_N);
        const uint32_t a_buf = a_base + (uint32_t)buf * A_BUF_BYTES;
        uint32_t acc = 0;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
          const int shift = HALO + (tap / 3 - 1) * 16 + (tap % 3 - 1);   // 0..34 rows into the halo tile
          if (it == 0) { rz::mbar_wait(bar_btap + 8 * tap, 0); rz::tc_fence_after(); }   // this tap's weights have landed
          // flags bit 4 (split input, c_in = 128 = [hi 0..63 | lo 0..63] of a 64-channel float32-accurate
          // activation against weights [Whi | Wlo]): three products per tap -- hi*Whi, lo*Whi, hi*Wlo
          const int n_prod = (p.flags & 16) ? 3 : p.kblocks;
          for (int pr = 0; pr < n_prod; ++pr) {
            const int ka = (p.flags & 16) ? (pr == 1 ? 1 : 0) : pr;      // k-block of the activation tile
            const int kw = (p.flags & 16) ? (pr == 2 ? 1 : 0) : pr;      // k-block of the weights
            const uint32_t a_addr = a_buf + (uint32_t)ka * A_KB_BYTES + (uint32_t)shift * 128u;
            const uint32_t b_addr = smem_base + (uint32_t)(tap * 2 + kw) * B_TILE_BYTES;
            const uint64_t adesc = rz::umma_desc_sw128_bo(a_addr, (p.flags & 1) ? (a_addr >> 7) & 7u : 0u);
            const uint64_t bdesc = rz::umma_desc_sw128(b_addr);
            // flags bit 7: only the first 96 of the 128 input channels carry data ([hi | lo | hi] of a 32-channel
            // pair layout; the fourth block would add the lo*lo products): skip the last two k-steps
            const int n_kk = ((p.flags & 128) && pr == 1) ? 2 : 4;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              if (kk < n_kk) {
                rz::umma_bf16_pair_pred(d_tmem, adesc + (uint64_t)(2 * kk), bdesc + (uint64_t)(2 * kk), idesc, acc, issue);
                acc = 1;
              }
            }
          }
        }
        // accumulator complete: both CTAs drain their half; the A buffers are recycled by the
        // epilogues, not here
        rz::umma_commit_pair_pred(bar_tfull + 8 * buf, 3, issue);
      }
    }
  } else if (!kHead) {
    // ===== epilogue warps 2..9: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4: one output
    // row x half the channels per thread.  Two warps per scheduler and half the serial work per thread:
    // with a single warp per quarter the epilogue (TMEM drain, bias/residual/ReLU, bf16 packing, staging)
    // took longer than the tile's 72 MMAs and set the pace of the kernel (profiles/r1_run24_*).
    // TMEM -> registers -> (+bias, +residual, ReLU, pad mask, bf16) -> 256-bit global stores straight
    // from registers (one full 32-byte sector per lane and instruction).  Nothing is staged in shared
    // memory, so the A buffer goes back to the producer (a_empty) as soon as the tile's MMAs are done:
    // the reload of the next-but-one tile starts one epilogue earlier and has a whole MMA period to land.
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    constexpr int HALF = ACC_N / 2;                 // columns per thread
    constexpr int NCHH = HALF / 32;                 // 32-column TMEM chunks per thread
    const int col0 = hsel * HALF;                   // first output channel of this thread
    // flags bit 3 (split output): the layer has 64 real output channels (accumulator columns 0..63);
    // the row leaves as [hi 0..63 | lo 0..63], hi = bf16(x), lo = bf16(x - hi): warps with hsel = 0 write the high
    // parts, their partners read the SAME columns and write the rounding residues
    const bool split_out = (p.flags & 8) != 0;
    const int csrc = split_out ? 0 : hsel * HALF;                    // first accumulator column this thread reads
    const int r_in_tile = q * 32 + lane;
    auto row_valid = [&](int item_) {
      const int pos_ = (row_of(item_) + r_in_tile) & 255;
      return ((pos_ & 15) < p.board_w) && ((pos_ >> 4) < p.board);
    };
    // residual segment of this thread's row, double-buffered in registers: the loads for tile i+1 are issued
    // while tile i is processed.  (With the loads at the top of their own iteration the epilogue -- usually
    // behind the MMAs, so the accumulator is already waiting -- paid their latency in the open: 77 % against
    // 94 % tensor-pipe activity for layers with / without a residual input, profiles/r1_run26_*.)
    uint32_t res[NCHH * 2][8], resn[NCHH * 2][8];
    bool next_res = false;
    auto load_res = [&](int item_) {
      next_res = p.residual != nullptr && row_valid(item_);
      if (next_res) {
        const __nv_bfloat16* rrow = p.residual + ((size_t)row_of(item_) + r_in_tile) * 128 + col0;
#pragma unroll
        for (int j = 0; j < NCHH * 2; ++j) rz::ld_global_v8_stream(rrow + j * 16, resn[j]);
      }
    };
    if (worker < p.n_items) load_res(worker);
    int it = 0;
    for (int item = worker; item < p.n_items; item += n_workers, ++it) {
      const int buf = it & 1;
      const int row0 = row_of(item);
      const size_t row = (size_t)row0 + r_in_tile;
      const bool valid = row_valid(item);
      const bool have_res = next_res;
      if (have_res) {
#pragma unroll
        for (int j = 0; j < NCHH * 2; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) res[j][e] = resn[j][e];
      }
      if (item + n_workers < p.n_items) load_res(item + n_workers); else next_res = false;
      rz::mbar_wait(bar_tfull + 8 * buf, (uint32_t)(it >> 1) & 1u);
      rz::tc_fence_after();
      if (p.flags & 4) {   // PROBE ONLY (scripts/conv_overhead_probe.py): no epilogue work at all -> MMA-side floor
        rz::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          rz::mbar_arrive_cluster_relaxed(rz::mapa_shared(bar_tempty + 8 * buf, 0));
          if (warp == 2) rz::mbar_arrive(bar_aempty + 8 * buf);
        }
        continue;
      }
      if (warp == 2 && lane == 0) rz::mbar_arrive(bar_aempty + 8 * buf);   // MMAs done: A tile is dead
      // all of this thread's accumulator columns in flight at once, one wait
      uint32_t acc[NCHH][32];
#pragma unroll
      for (int ch = 0; ch < NCHH; ++ch)
        rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * ACC_N + csrc + ch * 32), acc[ch]);
      rz::tmem_ld_wait();
      // accumulator drained: the MMA issuer may overwrite it (no memory payload -> relaxed)
      rz::tc_fence_before();
      __syncwarp();
      if (lane == 0) rz::mbar_arrive_cluster_relaxed(rz::mapa_shared(bar_tempty + 8 * buf, 0));
      const float4* bias4 = reinterpret_cast<const float4*>(s_bias + (split_out ? csrc : col0));
      uint32_t pair8[8];
#pragma unroll
      for (int ch = 0; ch < NCHH; ++ch) {
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
            packed[e] = p.relu ? rz::pack_bf16x2_relu(v0, v1) : rz::pack_bf16x2(v0, v1);
            if (split_out && hsel == 1) {      // the residue of the (ReLU'd) float32 value after its bf16 high part
              if (p.relu) { v0 = fmaxf(v0, 0.0f); v1 = fmaxf(v1, 0.0f); }
              packed[e] = rz::pack_bf16x2(v0 - __uint_as_float(packed[e] << 16), v1 - __uint_as_float(packed[e] & 0xffff0000u));
            }
            if (!valid) packed[e] = 0u;
          }
          if (p.flags & 64) {
            // float32 output (the training step of the reference's own network keeps conv3's activation and the data
            // gradients at accumulator precision): 8 channels = one 32-byte store
            uint32_t f8[8];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = j * 8 + e * 2;
              float v0 = __uint_as_float(acc[ch][c]) + bb[e * 2];
              float v1 = __uint_as_float(acc[ch][c + 1]) + bb[e * 2 + 1];
              if (p.relu) { v0 = fmaxf(v0, 0.0f); v1 = fmaxf(v1, 0.0f); }
              f8[e * 2] = valid ? __float_as_uint(v0) : 0u;
              f8[e * 2 + 1] = valid ? __float_as_uint(v1) : 0u;
            }
            rz::st_global_v8(reinterpret_cast<float*>(p.out) + row * 128 + col0 + ch * 32 + j * 8, f8);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) pair8[(j & 1) * 4 + e] = packed[e];
            if (j & 1) rz::st_global_v8(p.out + row * 128 + col0 + ch * 32 + (j - 1) * 8, pair8);
          }
        }
      }
    }
    // no bulk store is outstanding here, so this waits for nothing; dropping it changes the kernel's register
    // allocation, which wants a measured A/B of its own
    if (warp == 2 && lane == 0) rz::tma_store_wait_all();
  } else {
    // ===== fused-heads layer (kHead): the same 8 epilogue warps; every thread turns its 64 channels of a row
    // into bf16 activations (never stored) and 6 partial dot products with the heads' 1x1 filters; the warp
    // holding channels 64..127 hands its partial sums to its partner through the tile's A buffer (dead once the
    // MMAs are done), which adds them, applies ReLU and writes the 6 features.  Summation order = that of
    // rz_net_heads.cu's conv1x1_position, so the fused and the separate path agree bit for bit. =====
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int col0 = hsel * 64;
    const int r_in_tile = q * 32 + lane;
    const int pos = (row_of(worker) + r_in_tile) & 255;       // the same square in every tile (see above)
    const bool valid = ((pos & 15) < p.board_w) && ((pos >> 4) < p.board);
    const bool have_res = p.residual != nullptr && valid;
    uint32_t res[4][8], resn[4][8];                            // residual double-buffered in registers
    auto load_res = [&](int item_) {
      const __nv_bfloat16* rrow = p.residual + ((size_t)row_of(item_) + r_in_tile) * 128 + col0;
#pragma unroll
      for (int j = 0; j < 4; ++j) rz::ld_global_v8_stream(rrow + j * 16, resn[j]);
    };
    if (have_res && worker < p.n_items) load_res(worker);
    int it = 0;
    for (int item = worker; item < p.n_items; item += n_workers, ++it) {
      const int buf = it & 1;
      const int row0 = row_of(item);
      const size_t row = (size_t)row0 + r_in_tile;
      if (have_res) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) res[j][e] = resn[j][e];
        if (item + n_workers < p.n_items) load_res(item + n_workers);
      }
      rz::mbar_wait(bar_tfull + 8 * buf, (uint32_t)(it >> 1) & 1u);
      rz::tc_fence_after();
      if (warp == 2 && lane == 0) rz::mbar_arrive(bar_aempty + 8 * buf);   // MMAs done: the A tile is dead
      uint32_t acc[2][32];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch)
        rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * ACC_N + col0 + ch * 32), acc[ch]);
      rz::tmem_ld_wait();
      rz::tc_fence_before();
      __syncwarp();
      if (lane == 0) rz::mbar_arrive_cluster_relaxed(rz::mapa_shared(bar_tempty + 8 * buf, 0));
      float hacc[6];
#pragma unroll
      for (int f = 0; f < 6; ++f) hacc[f] = hsel == 0 ? head.b[f] : 0.0f;
      const float4* bias4 = reinterpret_cast<const float4*>(s_bias + col0);
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
            uint32_t pk = p.relu ? rz::pack_bf16x2_relu(v0, v1) : rz::pack_bf16x2(v0, v1);
            if (!valid) pk = 0u;
            // on the bf16-rounded activations, channels in ascending order; flags bit 5: on the float32
            // activations themselves (the float32-accurate path of the stock network)
            float r0 = __uint_as_float(pk << 16), r1 = __uint_as_float(pk & 0xffff0000u);
            if (p.flags & 32) {
              r0 = valid ? (p.relu ? fmaxf(v0, 0.0f) : v0) : 0.0f;
              r1 = valid ? (p.relu ? fmaxf(v1, 0.0f) : v1) : 0.0f;
            }
            const int cc = ch * 32 + c;                 // channel within this thread's half
#pragma unroll
            for (int f = 0; f < 6; ++f) {
              hacc[f] = fmaf(r1, head.w[f * 128 + col0 + cc + 1], fmaf(r0, head.w[f * 128 + col0 + cc], hacc[f]));
            }
          }
        }
      }
      // partial sums of channels 64..127 -> 8 spare TMEM columns of this lane quarter (slot = tile parity); the partner
      // warp of the quarter reads them back.  (They used to travel through the tile's A buffer, which therefore went
      // back to the producer only at the END of this epilogue: the reload of the next-but-one tile started late and the
      // layer took 60 us longer than a plain one, profiles/r2_run48_wave_timeline_8192.log.)
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
        float* fo = head.feat + (size_t)(row >> 8) * (6 * 256) + pos;
#pragma unroll
        for (int f = 0; f < 6; ++f) fo[f * 256] = fmaxf(hacc[f] + __uint_as_float(hv[f]), 0.0f);
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

template <bool kHead>
int launch(const CUtensorMap& ta, const CUtensorMap& tw, const CUtensorMap& to, const Conv2Params& p,
           const HeadTaps& head, int ctas, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(rz_conv3x3_tc2_kernel<kHead>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) { rz_set_error("rz_net_conv3x3_tc2: smem attribute: %s", cudaGetErrorString(e)); return -2; }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ctas);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1 + rz_pdl_attr(&attr[1]);
  cudaError_t e = cudaLaunchKernelEx(&cfg, rz_conv3x3_tc2_kernel<kHead>, ta, tw, to, p, head);
  if (e != cudaSuccess) { rz_set_error("rz_net_conv3x3_tc2: launch failed: %s", cudaGetErrorString(e)); return -2; }
  return 0;
}

}  // namespace

static int conv2_entry(const void* act_in, const void* weight, const float* bias, const void* residual,
                       void* act_out, int n_boards, int board_size, int board_cols, int c_in, int relu, int cta_group,
                       int flags, int n_ctas, const float* w1x1_host, const float* b1x1_host, float* feat,
                       void* stream) {
  RZ_REQUIRE(act_in && weight && bias, "rz_net_conv3x3_tc2: null argument");
  RZ_REQUIRE(n_boards >= 0, "rz_net_conv3x3_tc2: n_boards %d", n_boards);
  RZ_REQUIRE(board_size >= 1 && board_size <= 15, "rz_net_conv3x3_tc2: board_size %d not in [1,15]", board_size);
  RZ_REQUIRE(board_cols >= 1 && board_cols <= 15, "rz_net_conv3x3_tc2: board_cols %d not in [1,15]", board_cols);
  RZ_REQUIRE(c_in == 64 || c_in == 128, "rz_net_conv3x3_tc2: c_in %d (64 or 128)", c_in);
  RZ_REQUIRE(cta_group == 2, "rz_net_conv3x3_tc2: cta_group %d (the kernel runs on CTA pairs: 2)", cta_group);
  RZ_REQUIRE(act_in != act_out, "rz_net_conv3x3_tc2: in-place convolution is not supported");
  RZ_REQUIRE(!(flags & (8 | 16)) || c_in == 128, "rz_net_conv3x3_tc2: the split modes (flags 8 / 16) need c_in = 128");
  RZ_REQUIRE(!(flags & 256) || (flags & 8), "rz_net_conv3x3_tc2: N = 64 (flag 256) goes with the split output (flag 8)");
  RZ_REQUIRE(!(flags & 128) || !(flags & 16), "rz_net_conv3x3_tc2: flags 128 (96 input channels) and 16 (split input) exclude each other");
  RZ_REQUIRE(!(flags & 64) || (!(flags & 8) && !residual && !feat),
             "rz_net_conv3x3_tc2: float32 output (flag 64) needs no residual and no split output");
  if (n_boards == 0) return 0;
  static HeadTaps head;   // ~3 KB: filled per call, copied into the launch parameters
  CUtensorMap tmap_act, tmap_w, tmap_out;
  if (rz::make_tmap_2d(&tmap_act, act_in, (uint64_t)n_boards * 256, (uint64_t)c_in, A_ROWS)) return -1;
  if (rz::make_tmap_2d(&tmap_w, weight, (uint64_t)9 * 128, (uint64_t)c_in, 64)) return -1;
  // kHead launches store nothing through this map; it then describes the input tensor's rows
  if (rz::make_tmap_2d(&tmap_out, feat ? act_in : act_out, (uint64_t)n_boards * 256, feat ? (uint64_t)c_in : 128, TILE_M))
    return -1;
  Conv2Params p;
  p.bias = bias;
  p.residual = (const __nv_bfloat16*)residual;
  p.out = (__nv_bfloat16*)act_out;
  p.n_items = n_boards;
  p.board = board_size;
  p.board_w = board_cols;
  p.kblocks = c_in / 64;
  p.relu = relu;
  p.flags = flags;
  int ctas = n_ctas > 0 ? n_ctas : 148;
  ctas &= ~1;                                       // workers are CTA pairs
  if (ctas < 2) ctas = 2;
  if (ctas / 2 > p.n_items) ctas = 2 * p.n_items;   // every worker gets at least one item
  if (feat) {
    for (int i = 0; i < 6 * 128; ++i) head.w[i] = w1x1_host[i];
    for (int i = 0; i < 6; ++i) head.b[i] = b1x1_host[i];
    head.feat = feat;
    return launch<true>(tmap_act, tmap_w, tmap_out, p, head, ctas, (cudaStream_t)stream);
  }
  return launch<false>(tmap_act, tmap_w, tmap_out, p, head, ctas, (cudaStream_t)stream);
}

extern "C" int rz_net_conv3x3_tc2(const void* act_in, const void* weight, const float* bias,
                                  const void* residual, void* act_out, int n_boards, int board_size,
                                  int board_cols, int c_in, int relu, int cta_group, int flags, int n_ctas,
                                  void* stream) {
  RZ_REQUIRE(act_out, "rz_net_conv3x3_tc2: null output");
  return conv2_entry(act_in, weight, bias, residual, act_out, n_boards, board_size, board_cols, c_in, relu, cta_group, flags,
                     n_ctas, nullptr, nullptr, nullptr, stream);
}

extern "C" int rz_net_conv3x3_tc2_head_ex(const void* act_in, const void* weight, const float* bias,
                                          const void* residual, int n_boards, int board_size, int board_cols,
                                          int c_in, int relu, int flags, const float* w1x1_host,
                                          const float* b1x1_host, float* feat, int n_ctas, void* stream) {
  RZ_REQUIRE(w1x1_host && b1x1_host && feat, "rz_net_conv3x3_tc2_head_ex: null head argument");
  RZ_REQUIRE((flags & ~(16 | 32 | 512)) == 0, "rz_net_conv3x3_tc2_head_ex: flags %d (16 = split input, 32 = float32 features, 512 = static weights)", flags);
  return conv2_entry(act_in, weight, bias, residual, nullptr, n_boards, board_size, board_cols, c_in, relu, 2, flags, n_ctas,
                     w1x1_host, b1x1_host, feat, stream);
}
