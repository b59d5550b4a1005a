// Stand-alone probe (not part of the library): does keeping the trunk convolution's activations in L2 instead of
// HBM make it faster once the card runs at its power limit?
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I rlzero_b200/csrc -o conv_l2_probe \
//        scripts/probes/conv_l2_probe.cu -lcuda -ldl -lpthread
//
// conv_l2_probe_kernel<kL2> is a copy of rz_conv3x3_tc2_kernel<false> (rlzero_b200/csrc/rz_net_tc2.cu, the fused-heads
// branch left out).  Its one change is in row_of: with kL2 = true board `item` uses rows (item % 256) * 256, so all
// 8192 tiles read and write a 16 MB window and input, output and residual together stay in the 126 MB L2.  The MMAs
// and the epilogue are unchanged (several pairs then write the same rows with the same values: harmless here).
// kL2 = false is the stock kernel.
//
// Workload: one ResNet-10 trunk behind the stem, i.e. 20 back-to-back 128 -> 128 launches on 8192 boards of 15x15
// (flag 512, PDL on, 148 CTAs), the even-numbered ones adding a residual in place (the output buffer), as
// NativeForward runs them.  After a warm-up the two kernels alternate in blocks of `reps` trunks (ABBA order),
// timed with CUDA events; a host thread samples SM clock and board power through NVML every 20 ms, and each block
// reports the mean of the samples taken while it ran.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvml.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <mutex>
#include <thread>
#include <vector>

#include "rz_common.cuh"
#include "rz_tc.cuh"

void rz_set_error(const char* fmt, ...) { (void)fmt; }
bool rz_pdl_enabled() { return true; }
unsigned long long* rz_probe_buffer = nullptr;
namespace rz { void set_error_tmap(const char* what, int code) { fprintf(stderr, "%s (%d)\n", what, code); } }

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


template <bool kL2>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_l2_probe_kernel(const __grid_constant__ CUtensorMap tmap_act,
                      const __grid_constant__ CUtensorMap tmap_w,
                      const __grid_constant__ CUtensorMap tmap_out, const Conv2Params p) {
  constexpr int ACC_N = 128;                       // accumulator columns per buffer
  // fused-heads layer: 16 more columns (two slots of 8) carry the upper channel half's partial sums from one warp of a
  // lane quarter to the other; the allocation is a power of two
  constexpr int TMEM_COLS = 2 * ACC_N;
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
    return (kL2 ? (item & 255) : item) * 256 + (int)rank * TILE_M;   // THE probe change (kL2)
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
  } else {
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
  }

  rz::tc_fence_before();
  rz::cluster_sync_all();
  if (warp == 1) {
    rz::tc_fence_after();
    rz::tmem_dealloc_pair(tmem_base, TMEM_COLS);
  }
}

}  // namespace

__global__ void fill_bf16(__nv_bfloat16* p, size_t n, uint32_t seed, float scale) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t h = (uint32_t)i * 2654435761u ^ seed;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13; h *= 3266489917u; h ^= h >> 16;
    p[i] = __float2bfloat16(scale * ((float)(h & 0xffffu) / 32768.0f - 1.0f));
  }
}

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { \
  fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); exit(1); } } while (0)

// NVML through dlopen (the driver's library; no link-time dependency)
struct Nvml {
  nvmlDevice_t dev = nullptr;
  nvmlReturn_t (*clock)(nvmlDevice_t, nvmlClockType_t, unsigned int*) = nullptr;
  nvmlReturn_t (*power)(nvmlDevice_t, unsigned int*) = nullptr;
  bool ok = false;
  void init() {
    void* h = dlopen("libnvidia-ml.so.1", RTLD_NOW);
    if (!h) return;
    auto init_fn = (nvmlReturn_t(*)())dlsym(h, "nvmlInit_v2");
    auto by_index = (nvmlReturn_t(*)(unsigned, nvmlDevice_t*))dlsym(h, "nvmlDeviceGetHandleByIndex_v2");
    auto name_fn = (nvmlReturn_t(*)(nvmlDevice_t, char*, unsigned))dlsym(h, "nvmlDeviceGetName");
    auto limit_fn = (nvmlReturn_t(*)(nvmlDevice_t, unsigned*))dlsym(h, "nvmlDeviceGetEnforcedPowerLimit");
    auto maxclk_fn = (nvmlReturn_t(*)(nvmlDevice_t, nvmlClockType_t, unsigned*))dlsym(h, "nvmlDeviceGetMaxClockInfo");
    clock = (nvmlReturn_t(*)(nvmlDevice_t, nvmlClockType_t, unsigned*))dlsym(h, "nvmlDeviceGetClockInfo");
    power = (nvmlReturn_t(*)(nvmlDevice_t, unsigned*))dlsym(h, "nvmlDeviceGetPowerUsage");
    if (!init_fn || !by_index || !clock || !power || init_fn() != NVML_SUCCESS) return;
    int cu = 0;
    CK(cudaGetDevice(&cu));
    if (by_index((unsigned)cu, &dev) != NVML_SUCCESS) return;   // CUDA_VISIBLE_DEVICES unset on these runs
    char name[96] = {0};
    unsigned lim = 0, mx = 0;
    if (name_fn) name_fn(dev, name, sizeof(name));
    if (limit_fn) limit_fn(dev, &lim);
    if (maxclk_fn) maxclk_fn(dev, NVML_CLOCK_SM, &mx);
    printf("{\"nvml_device\": \"%s\", \"enforced_power_limit_w\": %.1f, \"sm_max_mhz\": %u}\n", name, lim / 1000.0, mx);
    ok = true;
  }
};

struct Sample { double t; unsigned mhz; unsigned mw; };

int main(int argc, char** argv) {
  const int n = argc > 1 ? atoi(argv[1]) : 8192;       // boards
  const int reps = argc > 2 ? atoi(argv[2]) : 50;      // trunks per timed block
  const int rounds = argc > 3 ? atoi(argv[3]) : 6;     // ABBA rounds: 2 blocks of each kernel per round
  const int n_layers = 20;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("{\"device\": \"%s\", \"sms\": %d, \"l2_mb\": %.1f, \"boards\": %d, \"reps_per_block\": %d, \"rounds\": %d}\n",
         prop.name, prop.multiProcessorCount, prop.l2CacheSize / 1048576.0, n, reps, rounds);
  Nvml nv;
  nv.init();

  const size_t rows = (size_t)n * 256;
  __nv_bfloat16 *buf[2], *w;
  float* bias;
  CK(cudaMalloc(&buf[0], rows * 128 * 2));
  CK(cudaMalloc(&buf[1], rows * 128 * 2));
  CK(cudaMalloc(&w, (size_t)n_layers * 9 * 128 * 128 * 2));
  CK(cudaMalloc(&bias, 128 * sizeof(float)));
  CK(cudaMemset(bias, 0, 128 * sizeof(float)));
  fill_bf16<<<1184, 256>>>(buf[0], rows * 128, 1u, 1.0f);
  fill_bf16<<<1184, 256>>>(buf[1], rows * 128, 2u, 1.0f);
  fill_bf16<<<1184, 256>>>(w, (size_t)n_layers * 9 * 128 * 128, 3u, 0.02f);
  CK(cudaDeviceSynchronize());

  CUtensorMap tm_in[2], tm_w[20], tm_out[2];
  for (int b = 0; b < 2; ++b) {
    if (rz::make_tmap_2d(&tm_in[b], buf[b], rows, 128, A_ROWS)) return 1;
    if (rz::make_tmap_2d(&tm_out[b], buf[b], rows, 128, TILE_M)) return 1;
  }
  for (int l = 0; l < n_layers; ++l)
    if (rz::make_tmap_2d(&tm_w[l], w + (size_t)l * 9 * 128 * 128, 9 * 128, 128, 64)) return 1;
  CK(cudaFuncSetAttribute(conv_l2_probe_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  CK(cudaFuncSetAttribute(conv_l2_probe_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  cudaStream_t st;
  CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));

  auto trunk = [&](bool l2) {
    int cur = 0;
    for (int l = 1; l <= n_layers; ++l) {
      Conv2Params p;
      p.bias = bias;
      p.residual = (l % 2 == 0) ? buf[1 - cur] : nullptr;   // in place: the block's residual is the output buffer
      p.out = buf[1 - cur];
      p.n_items = n;
      p.board = 15;
      p.board_w = 15;
      p.kblocks = 2;
      p.relu = 1;
      p.flags = 514;
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(148);
      cfg.blockDim = dim3(NUM_THREADS);
      cfg.dynamicSmemBytes = SMEM_BYTES;
      cfg.stream = st;
      cudaLaunchAttribute attr[2];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1 + rz_pdl_attr(&attr[1]);
      if (l2) CK(cudaLaunchKernelEx(&cfg, conv_l2_probe_kernel<true>, tm_in[cur], tm_w[l - 1], tm_out[1 - cur], p));
      else    CK(cudaLaunchKernelEx(&cfg, conv_l2_probe_kernel<false>, tm_in[cur], tm_w[l - 1], tm_out[1 - cur], p));
      cur = 1 - cur;
    }
  };

  std::vector<Sample> samples;
  std::mutex mu;
  std::atomic<bool> stop{false};
  const auto t0 = std::chrono::steady_clock::now();
  auto now_s = [&]() { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); };
  std::thread sampler([&]() {
    while (!stop.load()) {
      if (nv.ok) {
        unsigned mhz = 0, mw = 0;
        nv.clock(nv.dev, NVML_CLOCK_SM, &mhz);
        nv.power(nv.dev, &mw);
        std::lock_guard<std::mutex> g(mu);
        samples.push_back({now_s(), mhz, mw});
      }
      std::this_thread::sleep_for(std::chrono::milliseconds(20));
    }
  });

  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  // warm-up: both kernels, then long enough on the stock one for the card to settle at its power limit
  for (int r = 0; r < 20; ++r) { trunk(false); trunk(true); }
  for (int r = 0; r < 4 * reps; ++r) trunk(false);
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());

  std::vector<double> us[2], mhz[2], watt[2];
  for (int round = 0; round < rounds; ++round) {
    for (int k = 0; k < 2; ++k) {
      const bool l2 = (k == 0) == (round % 2 == 1);          // ABBA: stock first in even rounds
      const double ts = now_s();
      CK(cudaEventRecord(e0, st));
      for (int r = 0; r < reps; ++r) trunk(l2);
      CK(cudaEventRecord(e1, st));
      CK(cudaEventSynchronize(e1));
      const double te = now_s();
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, e0, e1));
      double sm = 0, sp = 0;
      int ns = 0;
      {
        std::lock_guard<std::mutex> g(mu);
        for (const Sample& s : samples)
          if (s.t >= ts && s.t <= te) { sm += s.mhz; sp += s.mw / 1000.0; ++ns; }
      }
      const double per_launch = 1000.0 * ms / (reps * n_layers);
      us[l2].push_back(per_launch);
      if (ns) { mhz[l2].push_back(sm / ns); watt[l2].push_back(sp / ns); }
      printf("{\"round\": %d, \"kernel\": \"%s\", \"trunk_ms\": %.4f, \"us_per_launch\": %.2f, \"sm_mhz_mean\": %.0f, "
             "\"power_w_mean\": %.1f, \"nvml_samples\": %d}\n",
             round, l2 ? "l2_window" : "stock", ms / reps, per_launch, ns ? sm / ns : 0.0, ns ? sp / ns : 0.0, ns);
      fflush(stdout);
    }
  }
  stop = true;
  sampler.join();
  CK(cudaGetLastError());
  auto median = [](std::vector<double> v) {
    if (v.empty()) return 0.0;
    std::sort(v.begin(), v.end());
    return v.size() % 2 ? v[v.size() / 2] : 0.5 * (v[v.size() / 2 - 1] + v[v.size() / 2]);
  };
  const double a = median(us[0]), b = median(us[1]);
  printf("{\"summary\": true, \"stock_us_per_launch_median\": %.2f, \"l2_us_per_launch_median\": %.2f, "
         "\"l2_faster_pct\": %.2f, \"stock_us_min_max\": [%.2f, %.2f], \"l2_us_min_max\": [%.2f, %.2f], "
         "\"stock_sm_mhz_median\": %.0f, \"l2_sm_mhz_median\": %.0f, \"stock_power_w_median\": %.1f, "
         "\"l2_power_w_median\": %.1f}\n",
         a, b, 100.0 * (a - b) / a, *std::min_element(us[0].begin(), us[0].end()),
         *std::max_element(us[0].begin(), us[0].end()), *std::min_element(us[1].begin(), us[1].end()),
         *std::max_element(us[1].begin(), us[1].end()), median(mhz[0]), median(mhz[1]), median(watt[0]),
         median(watt[1]));
  return 0;
}
