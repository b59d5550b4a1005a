// rlzero_b200 -- the whole residual trunk of ONE board in one launch (small-batch latency path).
//
// Reference op: the 3x3 convolution stack of the policy-value network between the first convolution and the heads
// (rlzero/games/gomoku/policy_value_net.py:36-38 for the reference's own three layers; the ResNet-N trunk of SURVEY.md
// section 7), evaluated for the one position a sequential search expands per playout
// (rlzero/mcts/alphazero_mcts.py:73-94, the loop tools/train_alphazero.py:81-90 runs).
//
// Why: the batched path launches one kernel per layer.  For a single board every layer then costs a launch, a TMEM
// allocation, 295 KB of weights fetched before the first MMA, 2.4 us of MMAs, an HBM round trip for the activation and a
// kernel-end flush: 8-10 us per layer, 160-210 us per ResNet-10 evaluation (profiles/r2_run35_g1_wave_launches.csv).
// Here a CTA pair (tcgen05 cta_group::2, the same 256 x 128 x 16 MMAs in the same order as rz_net_tc2.cu, so the
// results are bit-identical to the batched path) keeps the board's activation in shared memory for the whole trunk:
//   * two ping-pong halo tiles per CTA (128 positions + 17 halo rows each side, 128 channels, SW128 K-major); the
//     epilogue writes the next layer's A operand straight into them, and the 17 boundary rows also into the peer
//     CTA's tile through distributed shared memory (st.shared::cluster) -- no activation touches HBM;
//   * the residual input of a block's second convolution is read back from the tile it is about to overwrite;
//   * the weights of all layers stream through an 8-slot ring of taps (16 KB per CTA and tap), the producer running up
//     to 8 taps ahead across layer boundaries; they are static, so the stream starts before the grid dependency
//     resolves (programmatic dependent launch, rz_common.cuh);
//   * the last layer's epilogue applies the heads' 1x1 convolutions exactly as rz_net_conv3x3_tc2_head_ex does.
// One pair per board: n_boards pairs run side by side (up to 74 at once on 148 SMs).
#include <cuda_bf16.h>

#include "rz_common.cuh"
#include "rz_tc.cuh"

namespace {

constexpr int TILE_M = 128;
constexpr int HALO = 17;
constexpr int A_ROWS = TILE_M + 2 * HALO;         // 162
constexpr int A_KB_BYTES = A_ROWS * 128;          // one k-block (64 channels) of the halo tile
constexpr int A_BUF_BYTES = 2 * A_KB_BYTES;       // 41472
constexpr int B_TILE_BYTES = 64 * 128;            // 64 output channels x 64 input channels
constexpr int SLOT_BYTES = 2 * B_TILE_BYTES;      // one tap: both k-blocks
constexpr int N_SLOTS = 8;
constexpr int MAX_LAYERS = 24;
constexpr int OFF_A = N_SLOTS * SLOT_BYTES;                   // 131072
constexpr int OFF_BIAS = OFF_A + 2 * A_BUF_BYTES;             // 214016
constexpr int OFF_CTRL = OFF_BIAS + MAX_LAYERS * 512;         // 226304
constexpr int SMEM_BYTES = OFF_CTRL + 512;                    // 226816 <= 232448
constexpr int NUM_THREADS = 320;                  // producer warp, MMA warp, 8 epilogue warps

struct TrunkParams {
  const float* bias;               // [n_layers][128]
  int n_layers;
  int n_boards;
  int board, board_w;
  unsigned relu_mask, res_mask;    // bit l: ReLU after layer l / layer l adds the activation two layers back
  // the float32-accurate layers of the reference's own PolicyValueNet (mode 'tc32', rz_net_conv3x3_tc2 flags 8|256 / 16 / 32):
  unsigned n64_mask;               // bit l: 64 real output channels, N = 64 MMAs, the row leaves as [hi 0..63 | lo 0..63]
  unsigned split_in_mask;          // bit l: input [hi 0..63 | lo 0..63] against weights [Whi | Wlo]: hi*Whi + lo*Whi + hi*Wlo
  int head_f32;                    // the 1x1 head convolutions read the float32 activations, not their bf16 rounding
  unsigned long long* probe;       // timing probe (rz_debug_set_probe; null in production): 4 globaltimer stamps / layer
};



struct HeadTapsS {
  float w[6 * 128];                // [filter][channel]
  float b[6];
  float* feat;                     // [n_boards][6][256] float32, position index p = y*16 + x
};

__device__ __forceinline__ void ld_shared_v4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void st_cluster_v4(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(cluster_addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

__global__ void __launch_bounds__(NUM_THREADS, 1)
rz_trunk_small_kernel(const __grid_constant__ CUtensorMap tmap_act, const __grid_constant__ CUtensorMap tmap_w,
                      const TrunkParams p, const __grid_constant__ HeadTapsS head) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = rz::smem_u32(smem_raw);
  const uint32_t a_base = smem_base + OFF_A;
  const uint32_t ctrl = smem_base + OFF_CTRL;
  uint8_t* ctrl_ptr = smem_raw + OFF_CTRL;
  const uint32_t bar_wfull = ctrl, bar_wempty = ctrl + 64;          // [N_SLOTS] each
  const uint32_t bar_afull = ctrl + 128, bar_aready = ctrl + 136, bar_tfull = ctrl + 144;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ctrl_ptr + 160);
  const float* s_bias = reinterpret_cast<const float*>(smem_raw + OFF_BIAS);

  const int warp = rz::uniform_i32((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const uint32_t rank = rz::uniform_u32(rz::cluster_ctarank());
  const bool leader = rank == 0;
  const int board = blockIdx.x >> 1;
  const int L = p.n_layers;

  if (threadIdx.x == 0 && (smem_base & 1023u)) __trap();
  if (warp == 0 && lane == 0) {
    rz::tma_prefetch_desc(&tmap_act);
    rz::tma_prefetch_desc(&tmap_w);
    for (int s = 0; s < N_SLOTS; ++s) { rz::mbar_init(bar_wfull + 8 * s, 1); rz::mbar_init(bar_wempty + 8 * s, 1); }
    rz::mbar_init(bar_afull, 1);
    rz::mbar_init(bar_aready, 16);        // the 8 epilogue warps of both CTAs
    rz::mbar_init(bar_tfull, 1);
    rz::fence_barrier_init();
  }
  if (warp == 1) { rz::tmem_alloc_pair(rz::smem_u32(tmem_holder), 128); rz::tmem_relinquish_pair(); }
  // biases of all layers (static, like the weights: fetched before the grid dependency resolves)
  for (int i = threadIdx.x; i < L * 128; i += NUM_THREADS) reinterpret_cast<float*>(smem_raw + OFF_BIAS)[i] = p.bias[i];
  // halo bands of the second tile: zero = the padding above / below the board (the first tile's arrive with the TMA
  // load; between the bands every row is written by an epilogue thread before it is read)
  for (int i = threadIdx.x; i < 4 * HALO * 8; i += NUM_THREADS) {
    const int range = i / (HALO * 8), c = i % (HALO * 8);        // (k-block, band), 16-byte chunk within the band
    const uint32_t addr = a_base + A_BUF_BYTES + (uint32_t)(range >> 1) * A_KB_BYTES +
                          (uint32_t)((range & 1) ? (HALO + TILE_M) * 128 : 0) + (uint32_t)c * 16u;
    rz::st_shared_v4(addr, 0u, 0u, 0u, 0u);
  }
  fence_proxy_async_all();
  rz::tc_fence_before();
  rz::cluster_sync_all();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (threadIdx.x != 0) { rz::grid_dep_wait(); rz::grid_dep_launch(); }
  if (warp == 0) {
    // ===== producer: the weight taps of every layer through the ring; the board's halo tile once =====
    if (lane == 0) {
      const int total = L * 9;
      const int ahead = total < N_SLOTS ? total : N_SLOTS;
      for (int idx = 0; idx <= total; ++idx) {
        if (idx == ahead) {
          // the ring is full (or everything is requested): now the activation, which the previous kernel wrote
          rz::grid_dep_wait();
          rz::grid_dep_launch();
          const uint32_t l_afull = rz::mapa_shared(bar_afull, 0);
          if (leader) rz::mbar_expect_tx(bar_afull, (uint32_t)(2 * 2 * A_KB_BYTES));
          const int row0 = board * 256 + (int)rank * TILE_M - HALO;
          for (int kb = 0; kb < 2; ++kb)
            rz::tma_load_2d_pair(a_base + (uint32_t)kb * A_KB_BYTES, &tmap_act, l_afull, kb * 64, row0);
        }
        if (idx == total) break;
        const int slot = idx % N_SLOTS;
        if (idx >= N_SLOTS) rz::mbar_wait(bar_wempty + 8 * slot, ((uint32_t)(idx / N_SLOTS) - 1u) & 1u);
        const uint32_t l_full = rz::mapa_shared(bar_wfull + 8 * slot, 0);
        if (leader) rz::mbar_expect_tx(bar_wfull + 8 * slot, (uint32_t)(2 * SLOT_BYTES));
        const int layer = idx / 9, tap = idx % 9;
        for (int kb = 0; kb < 2; ++kb)
          rz::tma_load_2d_pair(smem_base + (uint32_t)slot * SLOT_BYTES + (uint32_t)kb * B_TILE_BYTES, &tmap_w, l_full,
                               kb * 64, layer * 1152 + tap * 128 + (int)rank * 64);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA; whole warp converged, one elected lane issues) =====
    if (leader) {
      constexpr uint32_t idesc = rz::umma_idesc_bf16(256, 128);
      const uint32_t issue = rz::elect_one();
      const uint32_t d_tmem = rz::uniform_u32(tmem_base);
      int idx = 0;
      for (int l = 0; l < L; ++l) {
        if (l == 0) rz::mbar_wait(bar_afull, 0);
        else        rz::mbar_wait(bar_aready, (uint32_t)(l - 1) & 1u);   // layer l-1 written in both CTAs, TMEM drained
        rz::tc_fence_after();
        if (p.probe && board == 0 && lane == 0) p.probe[l * 8 + 0] = rz::globaltimer_ns();
        const uint32_t a_buf = a_base + (uint32_t)(l & 1) * A_BUF_BYTES;
        const bool split_in = (p.split_in_mask >> l) & 1u;
        const uint32_t idesc_l = ((p.n64_mask >> l) & 1u) ? rz::umma_idesc_bf16(256, 64) : idesc;
        const int n_prod = split_in ? 3 : 2;
        uint32_t acc = 0;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap, ++idx) {
          const int slot = idx % N_SLOTS;
          const int shift = HALO + (tap / 3 - 1) * 16 + (tap % 3 - 1);
          rz::mbar_wait(bar_wfull + 8 * slot, (uint32_t)(idx / N_SLOTS) & 1u);
          rz::tc_fence_after();
          for (int pr = 0; pr < n_prod; ++pr) {
            const int ka = split_in ? (pr == 1 ? 1 : 0) : pr;      // k-block of the activation tile
            const int kw = split_in ? (pr == 2 ? 1 : 0) : pr;      // k-block of the weights
            const uint64_t adesc = rz::umma_desc_sw128(a_buf + (uint32_t)ka * A_KB_BYTES + (uint32_t)shift * 128u);
            const uint64_t bdesc = rz::umma_desc_sw128(smem_base + (uint32_t)slot * SLOT_BYTES + (uint32_t)kw * B_TILE_BYTES);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              rz::umma_bf16_pair_pred(d_tmem, adesc + (uint64_t)(2 * kk), bdesc + (uint64_t)(2 * kk), idesc_l, acc, issue);
              acc = 1;
            }
          }
          rz::umma_commit_pair_pred(bar_wempty + 8 * slot, 3, issue);     // both producers may refill this tap slot
        }
        rz::umma_commit_pair_pred(bar_tfull, 3, issue);                   // accumulator complete in both CTAs
        if (p.probe && board == 0 && lane == 0) p.probe[l * 8 + 1] = rz::globaltimer_ns();
      }
    }
  } else {
    // ===== epilogue warps 2..9: TMEM lane quarter = warp % 4, channel half (= k-block) = (warp - 2) / 4 =====
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int col0 = hsel * 64;
    const int r_in_tile = q * 32 + lane;
    const int pos = (int)rank * TILE_M + r_in_tile;
    const bool valid = ((pos & 15) < p.board_w) && ((pos >> 4) < p.board);
    // where this thread's 64 channels live in a halo tile (k-block hsel, row HALO + r), and in the peer's tile when the
    // row is one of the 17 next to the seam between the two CTAs
    const uint32_t row_off = (uint32_t)hsel * A_KB_BYTES + (uint32_t)(HALO + r_in_tile) * 128u;
    const bool seam = leader ? (r_in_tile >= TILE_M - HALO) : (r_in_tile < HALO);
    const int peer_row = leader ? (r_in_tile - (TILE_M - HALO)) : (HALO + TILE_M + r_in_tile);
    const uint32_t peer_off = (uint32_t)hsel * A_KB_BYTES + (uint32_t)peer_row * 128u;
    const uint32_t l_aready = rz::mapa_shared(bar_aready, 0);
    for (int l = 0; l < L; ++l) {
      const bool last = l == L - 1;
      const bool relu = (p.relu_mask >> l) & 1u;
      const bool have_res = ((p.res_mask >> l) & 1u) && valid;
      // 64-channel layer with split output: both column halves of the epilogue read accumulator columns 0..63; the
      // upper half's threads write the rounding residues of the (ReLU'd) float32 values after their bf16 high parts
      const bool split_out = (p.n64_mask >> l) & 1u;
      const int csrc = split_out ? 0 : col0;
      const uint32_t dst = a_base + (uint32_t)((l + 1) & 1) * A_BUF_BYTES;   // next layer's input = this layer's residual
      uint32_t res[8][4];
      if (have_res) {
        const uint32_t srow = dst + row_off;
        const uint32_t sw = (srow >> 7) & 7u;
#pragma unroll
        for (int j = 0; j < 8; ++j) ld_shared_v4(srow + (((uint32_t)j ^ sw) << 4), res[j]);
      }
      // this layer's 64 biases into registers while the MMAs still run (the epilogue is on the critical path of every
      // layer: nothing else overlaps it)
      float4 bias_r[16];
      {
        const float4* bias4 = reinterpret_cast<const float4*>(s_bias + l * 128 + csrc);
#pragma unroll
        for (int i = 0; i < 16; ++i) bias_r[i] = bias4[i];
      }
      rz::mbar_wait(bar_tfull, (uint32_t)l & 1u);
      rz::tc_fence_after();
      if (p.probe && board == 0 && leader && warp == 2 && lane == 0) p.probe[l * 8 + 2] = rz::globaltimer_ns();
      uint32_t acc[2][32];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch)
        rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(csrc + ch * 32), acc[ch]);
      rz::tmem_ld_wait();
      const bool stamp = p.probe && board == 0 && leader && warp == 2 && lane == 0;
      if (stamp) p.probe[l * 8 + 3] = rz::globaltimer_ns();
      if (!last) {
        const uint32_t srow = dst + row_off;
        const uint32_t sw = (srow >> 7) & 7u;
        const uint32_t prow = rz::mapa_shared(dst + peer_off, rank ^ 1u);
        const uint32_t psw = ((dst + peer_off) >> 7) & 7u;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 b0 = bias_r[ch * 8 + j * 2], b1 = bias_r[ch * 8 + j * 2 + 1];
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
            uint32_t packed[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = j * 8 + e * 2;
              float v0 = __uint_as_float(acc[ch][c]) + bb[e * 2];
              float v1 = __uint_as_float(acc[ch][c + 1]) + bb[e * 2 + 1];
              if (have_res) {
                const uint32_t rw = res[ch * 4 + j][e];
                v0 += __uint_as_float(rw << 16);
                v1 += __uint_as_float(rw & 0xffff0000u);
              }
              packed[e] = relu ? rz::pack_bf16x2_relu(v0, v1) : rz::pack_bf16x2(v0, v1);
              if (split_out && hsel == 1) {
                if (relu) { v0 = fmaxf(v0, 0.0f); v1 = fmaxf(v1, 0.0f); }
                packed[e] = rz::pack_bf16x2(v0 - __uint_as_float(packed[e] << 16), v1 - __uint_as_float(packed[e] & 0xffff0000u));
              }
              if (!valid) packed[e] = 0u;
            }
            const uint32_t chunk = (uint32_t)(ch * 4 + j);
            rz::st_shared_v4(srow + ((chunk ^ sw) << 4), packed[0], packed[1], packed[2], packed[3]);
            if (seam) st_cluster_v4(prow + ((chunk ^ psw) << 4), packed[0], packed[1], packed[2], packed[3]);
          }
        }
        // tile rows -> visible to the tensor core's (async proxy) reads of both CTAs, then "layer l is in place"
        if (stamp) p.probe[l * 8 + 4] = rz::globaltimer_ns();
        fence_proxy_async_all();
        if (stamp) p.probe[l * 8 + 5] = rz::globaltimer_ns();
        rz::tc_fence_before();
        __syncwarp();
        if (stamp) p.probe[l * 8 + 6] = rz::globaltimer_ns();
        if (lane == 0) rz::mbar_arrive_cluster(l_aready);
        if (p.probe && board == 0 && leader && warp == 2 && lane == 0) p.probe[l * 8 + 7] = rz::globaltimer_ns();
      } else {
        // the heads' 1x1 convolutions on the bf16-rounded activations of the last layer, as rz_net_conv3x3_tc2_head_ex:
        // channels in ascending order, the upper half's partial sums handed over through the (dead) input tile
        float hacc[6];
#pragma unroll
        for (int f = 0; f < 6; ++f) hacc[f] = hsel == 0 ? head.b[f] : 0.0f;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 b0 = bias_r[ch * 8 + j * 2], b1 = bias_r[ch * 8 + j * 2 + 1];
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = j * 8 + e * 2;
              float v0 = __uint_as_float(acc[ch][c]) + bb[e * 2];
              float v1 = __uint_as_float(acc[ch][c + 1]) + bb[e * 2 + 1];
              if (have_res) {
                const uint32_t rw = res[ch * 4 + j][e];
                v0 += __uint_as_float(rw << 16);
                v1 += __uint_as_float(rw & 0xffff0000u);
              }
              uint32_t pk = relu ? rz::pack_bf16x2_relu(v0, v1) : rz::pack_bf16x2(v0, v1);
              if (!valid) pk = 0u;
              float r0 = __uint_as_float(pk << 16), r1 = __uint_as_float(pk & 0xffff0000u);
              if (p.head_f32) {
                r0 = valid ? (relu ? fmaxf(v0, 0.0f) : v0) : 0.0f;
                r1 = valid ? (relu ? fmaxf(v1, 0.0f) : v1) : 0.0f;
              }
              const int cc = ch * 32 + c;
#pragma unroll
              for (int f = 0; f < 6; ++f)
                hacc[f] = fmaf(r1, head.w[f * 128 + col0 + cc + 1], fmaf(r0, head.w[f * 128 + col0 + cc], hacc[f]));
            }
          }
        }
        float* scratch = reinterpret_cast<float*>(smem_raw + OFF_A + (l & 1) * A_BUF_BYTES) + r_in_tile * 8;
        if (hsel == 1) {
#pragma unroll
          for (int f = 0; f < 6; ++f) scratch[f] = hacc[f];
        }
        rz::named_bar_sync(1, 256);
        if (hsel == 0) {
          float* fo = head.feat + (size_t)board * (6 * 256) + pos;
#pragma unroll
          for (int f = 0; f < 6; ++f) fo[f * 256] = fmaxf(hacc[f] + scratch[f], 0.0f);
        }
      }
    }
  }

  rz::tc_fence_before();
  rz::cluster_sync_all();
  if (warp == 1) {
    rz::tc_fence_after();
    rz::tmem_dealloc_pair(tmem_base, 128);
  }
}

}  // namespace

static int trunk_small_entry(const void* act_in, const void* weights, const float* biases, int n_layers,
                             unsigned relu_mask, unsigned res_mask, unsigned n64_mask, unsigned split_in_mask, int head_f32,
                             int n_boards, int board_size, int board_cols, const float* w1x1_host,
                             const float* b1x1_host, float* feat, void* stream) {
  RZ_REQUIRE(act_in && weights && biases && w1x1_host && b1x1_host && feat, "rz_net_trunk_small: null argument");
  RZ_REQUIRE(n_layers >= 1 && n_layers <= MAX_LAYERS, "rz_net_trunk_small: n_layers %d not in [1,%d]", n_layers, MAX_LAYERS);
  RZ_REQUIRE(n_boards >= 0, "rz_net_trunk_small: n_boards %d", n_boards);
  RZ_REQUIRE(board_size >= 1 && board_size <= 15, "rz_net_trunk_small: board_size %d not in [1,15]", board_size);
  RZ_REQUIRE(board_cols >= 1 && board_cols <= 15, "rz_net_trunk_small: board_cols %d not in [1,15]", board_cols);
  RZ_REQUIRE(!(res_mask & 1u), "rz_net_trunk_small: the first layer has no activation two layers back");
  if (n_boards == 0) return 0;
  static HeadTapsS head;
  CUtensorMap tmap_act, tmap_w;
  if (rz::make_tmap_2d(&tmap_act, act_in, (uint64_t)n_boards * 256, 128, A_ROWS)) return -1;
  if (rz::make_tmap_2d(&tmap_w, weights, (uint64_t)n_layers * 9 * 128, 128, 64)) return -1;
  TrunkParams p;
  p.bias = biases;
  p.n_layers = n_layers;
  p.n_boards = n_boards;
  p.board = board_size;
  p.board_w = board_cols;
  p.relu_mask = relu_mask;
  p.res_mask = res_mask;
  p.n64_mask = n64_mask;
  p.split_in_mask = split_in_mask;
  p.head_f32 = head_f32;
  p.probe = rz_probe_buffer;
  for (int i = 0; i < 6 * 128; ++i) head.w[i] = w1x1_host[i];
  for (int i = 0; i < 6; ++i) head.b[i] = b1x1_host[i];
  head.feat = feat;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(rz_trunk_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) { rz_set_error("rz_net_trunk_small: smem attribute: %s", cudaGetErrorString(e)); return -2; }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * n_boards));
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
  cudaError_t e = cudaLaunchKernelEx(&cfg, rz_trunk_small_kernel, tmap_act, tmap_w, p, head);
  if (e != cudaSuccess) { rz_set_error("rz_net_trunk_small: launch failed: %s", cudaGetErrorString(e)); return -2; }
  return 0;
}

extern "C" int rz_net_trunk_small(const void* act_in, const void* weights, const float* biases, int n_layers,
                                  unsigned relu_mask, unsigned res_mask, int n_boards, int board_size, int board_cols,
                                  const float* w1x1_host, const float* b1x1_host, float* feat, void* stream) {
  return trunk_small_entry(act_in, weights, biases, n_layers, relu_mask, res_mask, 0u, 0u, 0, n_boards, board_size, board_cols,
                           w1x1_host, b1x1_host, feat, stream);
}

// the same with the modes of the float32-accurate path of the reference's own PolicyValueNet (rz_net_conv3x3_tc2 flags
// 8 | 256: n64_mask, 16: split_in_mask, 32: head_f32): conv2 and conv3 + the 1x1 head convolutions in one launch
extern "C" int rz_net_trunk_small_ex(const void* act_in, const void* weights, const float* biases, int n_layers,
                                     unsigned relu_mask, unsigned res_mask, unsigned n64_mask, unsigned split_in_mask,
                                     int head_f32, int n_boards, int board_size, int board_cols,
                                     const float* w1x1_host, const float* b1x1_host, float* feat, void* stream) {
  RZ_REQUIRE(!(n64_mask & res_mask) && !(n64_mask >> (n_layers - 1) & 1u),
             "rz_net_trunk_small_ex: a 64-channel split-output layer has no skip input and is not the last layer");
  return trunk_small_entry(act_in, weights, biases, n_layers, relu_mask, res_mask, n64_mask, split_in_mask, head_f32,
                           n_boards, board_size, board_cols, w1x1_host, b1x1_host, feat, stream);
}
