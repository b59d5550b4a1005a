// rlzero_b200 -- 3x3 convolution of the policy-value trunk, revision 3: the data path of revision 2
// (rz_net_tc2.cu: weights resident in shared memory over a CTA pair, activation tile loaded once
// with its halo, row-shifted UMMA descriptors for the 9 taps, cta_group::2 MMAs) for ANY row
// stride of the padded position layout, so that 19x19 boards run on the tensor cores too.
//
// Reference op: nn.Conv2d(128, 128, 3, padding=1) (+ folded BatchNorm, residual, ReLU) of the
// trunk (rlzero/games/gomoku/policy_value_net.py:14-16,36-38; ResNet-N trunk of SURVEY.md 7;
// BASELINE.json config 4: 19x19 board, ResNet-20).
//
// Layout: act[row][c] bf16 with row = board*P + y*S + x, P = S*S, S = 16 (boards up to 15x15) or
// 20 (up to 19x19); squares with x >= W or y >= H hold zero, which gives every tap its halo (see
// rz_net_tc2.cu).  Tiles are 128 consecutive rows and need not be aligned to boards (P = 400 is not
// a multiple of 128); the tensor is padded to a multiple of 256 rows.
//
// What changes against revision 2, and why: the halo tile of stride 20 has 128 + 2*21 = 170 rows;
// two double-buffered 2-k-block tiles (87 KB) + the 147 KB of weights exceed the 227 KB of shared
// memory.  So
//   * the MMA loop runs k-block-outer (all 9 taps of input channels 0..63, then 64..127) and the
//     activation k-block tiles (170 x 128 B = 21.8 KB) cycle through a 3-slot ring: a slot is
//     released as soon as its 36 MMAs have completed, half a tile early, and refilled with the
//     next tile's data;
//   * the epilogue writes its rows straight from registers (256-bit global stores, as rev. 2's direct-store
//     epilogue; the 16 KB staging buffer of the first version is gone), which leaves room for a fourth ring slot at
//     strides 8 and 16.
// Shared memory: 147456 (weights) + 3*21760 (ring, stride 20) + 1024 = 213760 B; 4*20736 at stride 16: 231424 B.
#include <cuda_bf16.h>

#include "rz_common.cuh"
#include "rz_tc.cuh"

namespace {

constexpr int TILE_M = 128;
constexpr int B_TILE_BYTES = 64 * 128;            // 64 output channels x 64 input channels
constexpr int B_BYTES = 9 * 2 * B_TILE_BYTES;     // 147456
constexpr int NUM_THREADS = 320;    // producer warp, MMA warp, 8 epilogue warps (4 in the fused-heads layer)

template <int kS>
struct Geo {
  static constexpr int HALO = kS + 1;
  static constexpr int A_ROWS = TILE_M + 2 * HALO;
  static constexpr int SLOT_BYTES = A_ROWS * 128;
  static constexpr int P = kS * kS;
  static constexpr int OFF_RING = B_BYTES;
  static constexpr int N_SLOTS = (B_BYTES + 4 * SLOT_BYTES + 1024 <= 232448) ? 4 : 3;   // k-block halo tiles in flight
  static constexpr int OFF_CTRL = (OFF_RING + N_SLOTS * SLOT_BYTES + 127) / 128 * 128;
  static constexpr int SMEM = OFF_CTRL + 1024;
};

struct Conv3Params {
  const float* bias;               // [128]
  const __nv_bfloat16* residual;   // [rows][128] or null
  void* out;                       // [rows][128] bf16 (null in the fused-heads layer)
  int n_items;                     // pairs of 128-row tiles
  int total_rows;                  // n_boards * P (rows beyond it are padding)
  int H, W;
  int relu;
  int early_w;
};

struct HeadTaps3 {
  float w[6 * 128];                // [filter][channel]
  float b[6];
  float* feat;                     // [n_boards][6][P] float32
};

template <int kS, bool kHead>
__global__ void __launch_bounds__(NUM_THREADS, 1)
rz_conv3x3_tc3_kernel(const __grid_constant__ CUtensorMap tmap_act,
                      const __grid_constant__ CUtensorMap tmap_w,
                      const __grid_constant__ CUtensorMap tmap_out, const Conv3Params p,
                      const __grid_constant__ HeadTaps3 head) {
  using G = Geo<kS>;
  static_assert(G::SMEM <= 232448, "shared memory budget");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = rz::smem_u32(smem_raw);
  const uint32_t ring = smem_base + G::OFF_RING;
  const uint32_t ctrl = smem_base + G::OFF_CTRL;
  uint8_t* ctrl_ptr = smem_raw + G::OFF_CTRL;
  // weights: one barrier per (k-block, tap) at ctrl + 640 .. 783, loaded in the order the MMA loop consumes them and
  // right behind the first activation k-block, so the first tile starts after 16 KB of weights instead of 147 KB
  const uint32_t bar_btap = ctrl + 640, bar_afull = ctrl + 8, bar_aempty = ctrl + 40;   // [<= 4 slots] each
  const uint32_t bar_tfull = ctrl + 72, bar_tempty = ctrl + 88;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ctrl_ptr + 104);
  float* s_bias = reinterpret_cast<float*>(ctrl_ptr + 128);

  // warp index / cluster rank through a shuffle: provably warp-uniform, so the role branches are uniform and
  // the MMA issuer's operands live in uniform registers (see rz_tc.cuh, "warp-converged issue")
  const int warp = rz::uniform_i32((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const uint32_t rank = rz::uniform_u32(rz::cluster_ctarank());
  const bool leader = rank == 0;
  const int worker = blockIdx.x >> 1, n_workers = gridDim.x >> 1;

  // static weights (relu bit 1 of the entry points): weights and bias are fetched before the grid dependency resolves,
  // i.e. under the tail of the previous layer (rz_common.cuh, programmatic dependent launch)
  const bool early_w = p.early_w != 0;
  if (!early_w) rz::grid_dep_wait();
  if (threadIdx.x == 0 && (smem_base & 1023u)) __trap();
  if (warp == 0 && lane == 0) {
    rz::tma_prefetch_desc(&tmap_act);
    rz::tma_prefetch_desc(&tmap_w);
    rz::tma_prefetch_desc(&tmap_out);
    for (int j = 0; j < 18; ++j) rz::mbar_init(bar_btap + 8 * j, 1);
    for (int s = 0; s < G::N_SLOTS; ++s) {
      rz::mbar_init(bar_afull + 8 * s, 1);
      rz::mbar_init(bar_aempty + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      rz::mbar_init(bar_tfull + 8 * b, 1);
      rz::mbar_init(bar_tempty + 8 * b, 16);                 // the 8 epilogue warps of each CTA
    }
    rz::fence_barrier_init();
  }
  // (fused-heads layer: 16 more columns carry partial sums between the two warps of a lane quarter)
  if (warp == 1) { rz::tmem_alloc_pair(rz::smem_u32(tmem_holder), kHead ? 512 : 256); rz::tmem_relinquish_pair(); }
  if (threadIdx.x >= 64 && threadIdx.x < 192) s_bias[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  rz::tc_fence_before();
  rz::cluster_sync_all();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (early_w && threadIdx.x != 0) rz::grid_dep_wait();   // thread 0 (the producer) first requests the weights
  if (threadIdx.x != 0) rz::grid_dep_launch();
  if (warp == 0) {
    // ===== TMA producer: one (tile, k-block) halo tile per ring slot; the weights once, k-block-major, right behind
    // the first tile's two activation k-blocks =====
    if (lane == 0) {
      auto load_weights = [&](int kb) {
        for (int tap = 0; tap < 9; ++tap) {
          const uint32_t bar = bar_btap + 8 * (uint32_t)(kb * 9 + tap);
          if (leader) rz::mbar_expect_tx(bar, (uint32_t)(2 * B_TILE_BYTES));
          rz::tma_load_2d_pair(smem_base + (uint32_t)(tap * 2 + kb) * B_TILE_BYTES, &tmap_w, rz::mapa_shared(bar, 0),
                               kb * 64, tap * 128 + (int)rank * 64);
        }
      };
      if (early_w) { if (worker < p.n_items) { load_weights(0); load_weights(1); } rz::grid_dep_wait(); }
      rz::grid_dep_launch();
      int u = 0;   // running (tile, k-block) index
      for (int item = worker; item < p.n_items; item += n_workers) {
        const int row0 = item * 256 + (int)rank * TILE_M - G::HALO;
        for (int kb = 0; kb < 2; ++kb, ++u) {
          const int slot = u % G::N_SLOTS;
          rz::mbar_wait(bar_aempty + 8 * slot, ((uint32_t)(u / G::N_SLOTS) & 1u) ^ 1u);
          if (leader) rz::mbar_expect_tx(bar_afull + 8 * slot, (uint32_t)(2 * G::SLOT_BYTES));
          rz::tma_load_2d_pair(ring + (uint32_t)slot * G::SLOT_BYTES, &tmap_act,
                               rz::mapa_shared(bar_afull + 8 * slot, 0), kb * 64, row0);
          if (u < 2 && !early_w) load_weights(u);     // first tile only: k-block u's weights right behind its activations
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp of the leader CTA runs the loop converged; one elected lane issues =====
    if (leader) {
      constexpr uint32_t idesc = rz::umma_idesc_bf16(256, 128);
      const uint32_t issue = rz::elect_one();
      const uint32_t tmem_u = rz::uniform_u32(tmem_base);
      int it = 0, u = 0;
      for (int item = worker; item < p.n_items; item += n_workers, ++it) {
        const int buf = it & 1;
        rz::mbar_wait(bar_tempty + 8 * buf, ((uint32_t)(it >> 1) & 1u) ^ 1u);
        const uint32_t d_tmem = tmem_u + (uint32_t)(buf * 128);
        uint32_t acc = 0;
        for (int kb = 0; kb < 2; ++kb, ++u) {
          const int slot = u % G::N_SLOTS;
          rz::mbar_wait(bar_afull + 8 * slot, (uint32_t)(u / G::N_SLOTS) & 1u);
          rz::tc_fence_after();
          const uint32_t a_slot = ring + (uint32_t)slot * G::SLOT_BYTES;
#pragma unroll 1
          for (int tap = 0; tap < 9; ++tap) {
            const int shift = G::HALO + (tap / 3 - 1) * kS + (tap % 3 - 1);
            if (u < 2) { rz::mbar_wait(bar_btap + 8 * (uint32_t)(u * 9 + tap), 0); rz::tc_fence_after(); }
            const uint64_t adesc = rz::umma_desc_sw128(a_slot + (uint32_t)shift * 128u);
            const uint64_t bdesc = rz::umma_desc_sw128(smem_base + (uint32_t)(tap * 2 + kb) * B_TILE_BYTES);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              rz::umma_bf16_pair_pred(d_tmem, adesc + (uint64_t)(2 * kk), bdesc + (uint64_t)(2 * kk), idesc, acc, issue);
              acc = 1;
            }
          }
          rz::umma_commit_pair_pred(bar_aempty + 8 * slot, 3, issue);   // both CTAs may refill this ring slot
        }
        rz::umma_commit_pair_pred(bar_tfull + 8 * buf, 3, issue);       // accumulator complete in both CTAs
      }
    }
  } else if (!kHead) {
    // ===== epilogue warps 2..9: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4; one output row x
    // 64 channels per thread, written with 256-bit global stores straight from registers (rz_net_tc2.cu) =====
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int col0 = hsel * 64;
    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out);
    const int r_in_tile = q * 32 + lane;
    auto row_valid = [&](int row_) {
      const int board_ = row_ / G::P, pos_ = row_ - board_ * G::P;
      const int y_ = pos_ / kS, x_ = pos_ - y_ * kS;
      return row_ < p.total_rows && x_ < p.W && y_ < p.H;
    };
    // residual segment double-buffered in registers: tile i+1's loads fly while tile i is processed
    uint32_t res[4][8], resn[4][8];
    bool next_res = false;
    auto load_res = [&](int item_) {
      const int row_ = item_ * 256 + (int)rank * TILE_M + r_in_tile;
      next_res = p.residual != nullptr && row_valid(row_);
      if (next_res) {
        const __nv_bfloat16* rrow = p.residual + (size_t)row_ * 128 + col0;
#pragma unroll
        for (int j = 0; j < 4; ++j) rz::ld_global_v8_stream(rrow + j * 16, resn[j]);
      }
    };
    if (worker < p.n_items) load_res(worker);
    int it = 0;
    for (int item = worker; item < p.n_items; item += n_workers, ++it) {
      const int buf = it & 1;
      const int row0 = item * 256 + (int)rank * TILE_M;
      const int row = row0 + r_in_tile;
      const bool valid = row_valid(row);
      const bool have_res = next_res;
      if (have_res) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) res[j][e] = resn[j][e];
      }
      if (item + n_workers < p.n_items) load_res(item + n_workers); else next_res = false;
      rz::mbar_wait(bar_tfull + 8 * buf, (uint32_t)(it >> 1) & 1u);
      rz::tc_fence_after();
      uint32_t acc[2][32];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch)
        rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 128 + col0 + ch * 32), acc[ch]);
      rz::tmem_ld_wait();
      rz::tc_fence_before();
      __syncwarp();
      if (lane == 0) rz::mbar_arrive_cluster_relaxed(rz::mapa_shared(bar_tempty + 8 * buf, 0));
      const float4* bias4 = reinterpret_cast<const float4*>(s_bias + col0);
      uint32_t pair8[8];
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
            pair8[(j & 1) * 4 + e] = pk;
          }
          if (j & 1) rz::st_global_v8(out + (size_t)row * 128 + col0 + ch * 32 + (j - 1) * 8, pair8);
        }
      }
    }
  } else {
    // ===== fused-heads layer: the same 8 epilogue warps (TMEM lane quarter = warp % 4, channel half = (warp - 2) / 4).
    // Every thread turns its 64 channels of a row into bf16 activations (never stored) and 6 partial dot products with the
    // heads' 1x1 filters; the warp holding channels 64..127 hands its sums to its partner of the same lane quarter
    // through 8 spare TMEM columns (slot = tile parity), which adds them, applies ReLU and writes the 6 features.
    // Summation order = rz_net_heads.cu's conv1x1_position: channels 0..63 onto the bias, 64..127 onto zero.  (Until
    // round 2 four warps did all 128 channels of a row each -- 1536 FFMAs per thread and tile: the layer took 75 us
    // against 50 us for a plain one at Connect Four's size, profiles/r2_run51_wave_timeline_c4.log.)
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int col0 = hsel * 64;
    const int r_in_tile = q * 32 + lane;
    auto row_valid = [&](int row_) {
      const int board_ = row_ / G::P, pos_ = row_ - board_ * G::P;
      const int y_ = pos_ / kS, x_ = pos_ - y_ * kS;
      return row_ < p.total_rows && x_ < p.W && y_ < p.H;
    };
    uint32_t res[4][8], resn[4][8];
    bool next_res = false;
    auto load_res = [&](int item_) {
      const int row_ = item_ * 256 + (int)rank * TILE_M + r_in_tile;
      next_res = p.residual != nullptr && row_valid(row_);
      if (next_res) {
        const __nv_bfloat16* rrow = p.residual + (size_t)row_ * 128 + col0;
#pragma unroll
        for (int j = 0; j < 4; ++j) rz::ld_global_v8_stream(rrow + j * 16, resn[j]);
      }
    };
    if (worker < p.n_items) load_res(worker);
    int it = 0;
    for (int item = worker; item < p.n_items; item += n_workers, ++it) {
      const int buf = it & 1;
      const int row = item * 256 + (int)rank * TILE_M + r_in_tile;
      const int board = row / G::P, pos = row - board * G::P;
      const bool in_tensor = row < p.total_rows;
      const bool valid = row_valid(row);
      const bool have_res = next_res;
      if (have_res) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) res[j][e] = resn[j][e];
      }
      if (item + n_workers < p.n_items) load_res(item + n_workers); else next_res = false;
      rz::mbar_wait(bar_tfull + 8 * buf, (uint32_t)(it >> 1) & 1u);
      rz::tc_fence_after();
      uint32_t acc[2][32];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch)
        rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 128 + col0 + ch * 32), acc[ch]);
      rz::tmem_ld_wait();
      rz::tc_fence_before();
      __syncwarp();
      if (lane == 0) rz::mbar_arrive_cluster_relaxed(rz::mapa_shared(bar_tempty + 8 * buf, 0));
      float hacc[6];
#pragma unroll
      for (int f = 0; f < 6; ++f) hacc[f] = hsel == 0 ? head.b[f] : 0.0f;
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c = j * 8 + e * 2;
            float v0 = __uint_as_float(acc[ch][c]) + s_bias[col0 + ch * 32 + c];
            float v1 = __uint_as_float(acc[ch][c + 1]) + s_bias[col0 + ch * 32 + c + 1];
            if (have_res) {
              const uint32_t rw = res[ch * 2 + (j >> 1)][(j & 1) * 4 + e];
              v0 += __uint_as_float(rw << 16);
              v1 += __uint_as_float(rw & 0xffff0000u);
            }
            if (p.relu) { v0 = fmaxf(v0, 0.0f); v1 = fmaxf(v1, 0.0f); }
            if (!valid) { v0 = 0.0f; v1 = 0.0f; }
            const __nv_bfloat162 o2 = __floats2bfloat162_rn(v0, v1);
            const uint32_t pk = *reinterpret_cast<const uint32_t*>(&o2);
            const float r0 = __uint_as_float(pk << 16), r1 = __uint_as_float(pk & 0xffff0000u);
            const int cc = col0 + ch * 32 + c;
#pragma unroll
            for (int f = 0; f < 6; ++f)
              hacc[f] = fmaf(r1, head.w[f * 128 + cc + 1], fmaf(r0, head.w[f * 128 + cc], hacc[f]));
          }
        }
      }
      const uint32_t t_scr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(256 + buf * 8);
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
        if (in_tensor) {
          float* fo = head.feat + (size_t)board * (6 * G::P) + pos;
#pragma unroll
          for (int f = 0; f < 6; ++f) fo[f * G::P] = fmaxf(hacc[f] + __uint_as_float(hv[f]), 0.0f);
        }
      }
    }
  }

  rz::tc_fence_before();
  rz::cluster_sync_all();
  if (warp == 1) {
    rz::tc_fence_after();
    rz::tmem_dealloc_pair(tmem_base, kHead ? 512 : 256);
  }
}

template <int kS, bool kHead>
int launch3(const CUtensorMap& ta, const CUtensorMap& tw, const CUtensorMap& to, const Conv3Params& p,
            const HeadTaps3& head, int ctas, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(rz_conv3x3_tc3_kernel<kS, kHead>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Geo<kS>::SMEM);
    if (e != cudaSuccess) { rz_set_error("rz_net_conv3x3_tc3: smem attribute: %s", cudaGetErrorString(e)); return -2; }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ctas);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = Geo<kS>::SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1 + rz_pdl_attr(&attr[1]);
  cudaError_t e = cudaLaunchKernelEx(&cfg, rz_conv3x3_tc3_kernel<kS, kHead>, ta, tw, to, p, head);
  if (e != cudaSuccess) { rz_set_error("rz_net_conv3x3_tc3: launch failed: %s", cudaGetErrorString(e)); return -2; }
  return 0;
}

}  // namespace

// act_in / act_out / residual: bf16 [rows_alloc][128] with rows_alloc = round_up(n_boards * S*S, 256)
static int conv3_entry(const void* act_in, const void* weight, const float* bias, const void* residual,
                       void* act_out, int n_boards, int board_rows, int board_cols, int row_stride, int relu,
                       int n_ctas, const float* w1x1_host, const float* b1x1_host, float* feat, void* stream) {
  RZ_REQUIRE(act_in && weight && bias, "rz_net_conv3x3_tc3: null argument");
  RZ_REQUIRE(n_boards >= 0, "rz_net_conv3x3_tc3: n_boards %d", n_boards);
  RZ_REQUIRE(row_stride == 8 || row_stride == 16 || row_stride == 20, "rz_net_conv3x3_tc3: row_stride %d (8, 16 or 20)",
             row_stride);
  RZ_REQUIRE(board_rows >= 1 && board_rows < row_stride && board_cols >= 1 && board_cols < row_stride,
             "rz_net_conv3x3_tc3: board %dx%d does not fit row stride %d", board_rows, board_cols, row_stride);
  RZ_REQUIRE(act_in != act_out, "rz_net_conv3x3_tc3: in-place convolution is not supported");
  if (n_boards == 0) return 0;
  const long long total = (long long)n_boards * row_stride * row_stride;
  const long long rows_alloc = (total + 255) / 256 * 256;
  static HeadTaps3 head;
  CUtensorMap tmap_act, tmap_w, tmap_out;
  const uint32_t a_rows = TILE_M + 2 * (row_stride + 1);
  if (rz::make_tmap_2d(&tmap_act, act_in, (uint64_t)rows_alloc, 128, a_rows)) return -1;
  if (rz::make_tmap_2d(&tmap_w, weight, (uint64_t)9 * 128, 128, 64)) return -1;
  if (rz::make_tmap_2d(&tmap_out, feat ? act_in : act_out, (uint64_t)rows_alloc, 128, TILE_M)) return -1;
  Conv3Params p;
  p.bias = bias;
  p.residual = (const __nv_bfloat16*)residual;
  p.out = act_out;
  p.n_items = (int)(rows_alloc / 256);
  p.total_rows = (int)total;
  p.H = board_rows;
  p.W = board_cols;
  p.relu = relu & 1;
  p.early_w = (relu >> 1) & 1;
  int ctas = n_ctas > 0 ? n_ctas : 148;
  ctas &= ~1;
  if (ctas < 2) ctas = 2;
  if (ctas / 2 > p.n_items) ctas = 2 * p.n_items;
  cudaStream_t st = (cudaStream_t)stream;
  if (feat) {
    for (int i = 0; i < 6 * 128; ++i) head.w[i] = w1x1_host[i];
    for (int i = 0; i < 6; ++i) head.b[i] = b1x1_host[i];
    head.feat = feat;
    return row_stride == 8    ? launch3<8, true>(tmap_act, tmap_w, tmap_out, p, head, ctas, st)
           : row_stride == 16 ? launch3<16, true>(tmap_act, tmap_w, tmap_out, p, head, ctas, st)
                              : launch3<20, true>(tmap_act, tmap_w, tmap_out, p, head, ctas, st);
  }
  return row_stride == 8    ? launch3<8, false>(tmap_act, tmap_w, tmap_out, p, head, ctas, st)
         : row_stride == 16 ? launch3<16, false>(tmap_act, tmap_w, tmap_out, p, head, ctas, st)
                            : launch3<20, false>(tmap_act, tmap_w, tmap_out, p, head, ctas, st);
}

extern "C" int rz_net_conv3x3_tc3(const void* act_in, const void* weight, const float* bias,
                                  const void* residual, void* act_out, int n_boards, int board_rows,
                                  int board_cols, int row_stride, int relu, int n_ctas, void* stream) {
  RZ_REQUIRE(act_out, "rz_net_conv3x3_tc3: null output");
  return conv3_entry(act_in, weight, bias, residual, act_out, n_boards, board_rows, board_cols, row_stride, relu,
                     n_ctas, nullptr, nullptr, nullptr, stream);
}

extern "C" int rz_net_conv3x3_tc3_head(const void* act_in, const void* weight, const float* bias,
                                       const void* residual, int n_boards, int board_rows, int board_cols,
                                       int row_stride, int relu, const float* w1x1_host,
                                       const float* b1x1_host, float* feat, int n_ctas, void* stream) {
  RZ_REQUIRE(w1x1_host && b1x1_host && feat, "rz_net_conv3x3_tc3_head: null head argument");
  return conv3_entry(act_in, weight, bias, residual, nullptr, n_boards, board_rows, board_cols, row_stride, relu,
                     n_ctas, w1x1_host, b1x1_host, feat, stream);
}
