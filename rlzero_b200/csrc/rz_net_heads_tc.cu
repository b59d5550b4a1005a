// rlzero_b200 -- the fully connected layers of the policy / value heads on the tensor cores.
//
// Reference ops (rlzero/games/gomoku/policy_value_net.py): act_fc1 (4HW -> A) + log_softmax (:42-44),
// val_fc1 (2HW -> 64) + ReLU, val_fc2 (64 -> 1), tanh (:48-51), applied to the 6 head features per square
// that the last trunk layer's epilogue (rz_net_conv3x3_tc2_head_ex / _tc3_head) or rz_net_head_features wrote.
//
// The CUDA-core heads kernel (rz_net_heads.cu) spends 211 us on 8192 boards of 15x15 (3.8 GFLOP of fp32 FMAs
// through shared memory) and 721 us at 19x19.  Here the two FCs are one GEMM per 128 boards:
//   M = 128 boards, K = the 6*P features of a board in the PADDED square order k' = f*P + y*S + x -- exactly the
//       row feat[b][.] the trunk wrote, so building the A operand is a contiguous copy, and the weight matrix
//       carries zeros at the padding squares;
//   N = AS policy outputs for k' < 4P (filters 0..3), 64 value-hidden outputs for 4P <= k' < 6P (filters 4, 5).
// float32 accuracy on the bf16 tensor pipe: features and weights are split x = hi + lo (two bf16, lo = the
// rounding error of hi), and every k-step issues hi*hi + lo*hi + hi*lo (the dropped lo*lo term is 2^-18
// relative), so logits agree with the fp32 FC to ~1e-6 -- far inside the 1e-3 budget of the bf16 trunk.
// Accumulators live in TMEM: columns [0, AS) policy logits, [AS, AS+64) value hidden units; the epilogue
// (one thread per board row) adds the biases, does log_softmax / ReLU-FC2-tanh straight from TMEM.
#include <cuda_bf16.h>

#include "rz_common.cuh"
#include "rz_tc.cuh"

namespace {

constexpr int HT_THREADS = 256;
constexpr int HT_A_BYTES = 128 * 128;            // [128 boards][64 k] bf16, SW128
constexpr int HT_CTRL_BYTES = 2304;           // barriers, TMEM holder, biases [384 + 64 + 64] float

struct HeadsTcParams {
  const float* feat;      // [n][6][P]
  const float* bp;        // [AS]
  const float* bv1;       // [64]
  const float* wv2;       // [64]
  const float* bv2;       // [1]
  float* logp;            // [n][AS]
  float* value;           // [n]
  int n_boards, A, AS, P;
  int n_wslots;           // weight ring slots (2..4)
  int live_per_plane;     // cluster kernel: 64-feature chunks of a plane that hold real squares (the rest is zero padding)
  int w_box;              // rows per TMA box of the policy weights (divides AS)
  int tmem_cols;          // power of two >= AS + 64
  unsigned long long* probe;   // timing probe (rz_debug_set_probe; null in production): 8 stamps per chunk of CTA 0
};

// shared memory: A_hi | A_lo (one chunk of 64 features for 128 boards) | weight ring, slot = W_hi [WR rows] | W_lo [WR
// rows], WR = max(AS, 64) (the value chunks load 64 rows) | control
__host__ __device__ __forceinline__ uint32_t ht_w_rows(int AS) { return (uint32_t)(AS > 64 ? AS : 64); }
__host__ __device__ __forceinline__ uint32_t ht_slot_bytes(int AS) { return 2u * ht_w_rows(AS) * 128u; }

__global__ void __launch_bounds__(HT_THREADS, 1)
rz_heads_tc_kernel(const __grid_constant__ CUtensorMap tmap_whi, const __grid_constant__ CUtensorMap tmap_wlo,
                   const __grid_constant__ CUtensorMap tmap_vhi, const __grid_constant__ CUtensorMap tmap_vlo,
                   const HeadsTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = rz::smem_u32(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int AS = p.AS, P = p.P;
  const uint32_t slot_bytes = ht_slot_bytes(AS);
  const uint32_t a_hi = base, a_lo = base + HT_A_BYTES, w_ring = base + 2 * HT_A_BYTES;
  const uint32_t ctrl = w_ring + (uint32_t)p.n_wslots * slot_bytes;
  uint8_t* ctrl_ptr = smem_raw + (ctrl - base);
  const uint32_t bar_w = ctrl, bar_afree = ctrl + 32, bar_done = ctrl + 40;   // [4], [1], [1]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ctrl_ptr + 48);
  float* s_bp = reinterpret_cast<float*>(ctrl_ptr + 64);        // [AS <= 384]
  float* s_bv1 = s_bp + 384;                                    // [64]
  float* s_wv2 = s_bv1 + 64;                                    // [64]

  const int b0 = blockIdx.x * 128;
  const int r = tid & 127, khalf = tid >> 7;          // this thread builds row r, k in [32*khalf, 32*khalf + 32)
  const bool row_live = b0 + r < p.n_boards;
  const int K6 = 6 * P, K4 = 4 * P;
  const int n_chunks = (K6 + 63) >> 6, n_pol = K4 >> 6;   // 4P is a multiple of 64 for S in {8, 16, 20}

  // weights of chunk c into ring slot c % n_wslots (thread 0).  The weights are static (packed at refresh_weights),
  // so the first slots are requested before the grid dependency resolves; afterwards slot (c - 1) % n is refilled
  // with chunk c - 1 + n as soon as the MMAs of chunk c - 1 are done: the loads run n - 1 chunks ahead of the MMAs.
  // (With two stages of A + W and the load of chunk c requested in iteration c the L2 latency of 64 KB sat between
  // the conversion and the MMAs of every chunk: 66 us for ONE board, 84 us for 8192 -- profiles/r2_run35_*, run38.)
  auto issue_w = [&](int c) {
    const int s = c % p.n_wslots;
    const uint32_t w_hi = w_ring + (uint32_t)s * slot_bytes, w_lo = w_hi + ht_w_rows(AS) * 128u;
    if (c < n_pol) {
      rz::mbar_expect_tx(bar_w + 8 * s, 2u * (uint32_t)AS * 128u);
      for (int j = 0; j < AS; j += p.w_box) {
        rz::tma_load_2d(w_hi + (uint32_t)j * 128u, &tmap_whi, bar_w + 8 * s, c * 64, j);
        rz::tma_load_2d(w_lo + (uint32_t)j * 128u, &tmap_wlo, bar_w + 8 * s, c * 64, j);
      }
    } else {
      rz::mbar_expect_tx(bar_w + 8 * s, 2u * 64u * 128u);
      rz::tma_load_2d(w_hi, &tmap_vhi, bar_w + 8 * s, c * 64, 0);
      rz::tma_load_2d(w_lo, &tmap_vlo, bar_w + 8 * s, c * 64, 0);
    }
  };

  if (tid == 0) {
    if (base & 1023u) __trap();
    rz::tma_prefetch_desc(&tmap_whi);
    rz::tma_prefetch_desc(&tmap_wlo);
    rz::tma_prefetch_desc(&tmap_vhi);
    rz::tma_prefetch_desc(&tmap_vlo);
    for (int s = 0; s < 4; ++s) rz::mbar_init(bar_w + 8 * s, 1);
    rz::mbar_init(bar_afree, 1);
    rz::mbar_init(bar_done, 1);
    rz::fence_barrier_init();
    for (int c = 0; c < p.n_wslots && c < n_chunks; ++c) issue_w(c);
  }
  if (warp == 0) { rz::tmem_alloc(rz::smem_u32(tmem_holder), (uint32_t)p.tmem_cols); rz::tmem_relinquish(); }
  for (int i = tid; i < AS; i += HT_THREADS) s_bp[i] = i < p.A ? p.bp[i] : 0.0f;
  if (tid < 64) { s_bv1[tid] = p.bv1[tid]; s_wv2[tid] = p.wv2[tid]; }
  rz::grid_dep_wait();     // programmatic dependent launch (rz_common.cuh): the features come from the previous kernel
  rz::grid_dep_launch();
  rz::tc_fence_before();
  __syncthreads();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  const float* frow = p.feat + (size_t)(b0 + r) * K6 + 32 * khalf;
  // features: two chunks of look-ahead in registers (the loads of chunk c + 2 are issued while chunk c is converted)
  float4 pre[2][8];
  auto prefetch = [&](int c, float4 (&dst)[8]) {
    const int k0 = c * 64 + 32 * khalf;
    const bool live = row_live && c < n_chunks && k0 < K6;   // K6 is a multiple of 32
    const float4* src = reinterpret_cast<const float4*>(frow + (size_t)c * 64);
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[j] = live ? __ldg(src + j) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  };
  prefetch(0, pre[0]);
  prefetch(1, pre[1]);

  const uint32_t idesc_v = rz::umma_idesc_bf16(128, 64);
  auto step = [&](const int c, float4 (&cur)[8]) {
    const int s = c % p.n_wslots;
    const uint32_t w_hi = w_ring + (uint32_t)s * slot_bytes, w_lo = w_hi + ht_w_rows(AS) * 128u;
    const bool policy = c < n_pol;
    const bool stamp = p.probe && blockIdx.x == 0 && tid == 0;
    if (stamp) p.probe[c * 8 + 0] = rz::globaltimer_ns();
    if (c > 0) {
      // the MMAs of chunk c - 1 have read the A tile and their weight slot: convert into the one, refill the other
      rz::mbar_wait(bar_afree, (uint32_t)(c - 1) & 1u);
      if (stamp) p.probe[c * 8 + 1] = rz::globaltimer_ns();
      if (tid == 0 && c - 1 + p.n_wslots < n_chunks) issue_w(c - 1 + p.n_wslots);
    }
    // this thread's 32 features -> hi / lo bf16, 4 + 4 swizzled 16-byte chunks of row r
    {
      const uint32_t row_off = (uint32_t)r * 128u;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float x[8] = {cur[2 * q].x, cur[2 * q].y, cur[2 * q].z, cur[2 * q].w,
                            cur[2 * q + 1].x, cur[2 * q + 1].y, cur[2 * q + 1].z, cur[2 * q + 1].w};
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * e]), h1 = __float2bfloat16_rn(x[2 * e + 1]);
          hi[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
          lo[e] = rz::pack_bf16x2(x[2 * e] - __bfloat162float(h0), x[2 * e + 1] - __bfloat162float(h1));
        }
        const uint32_t chunk = (uint32_t)(khalf * 4 + q);
        const uint32_t off = row_off + ((chunk ^ ((uint32_t)r & 7u)) << 4);
        rz::st_shared_v4(a_hi + off, hi[0], hi[1], hi[2], hi[3]);
        rz::st_shared_v4(a_lo + off, lo[0], lo[1], lo[2], lo[3]);
      }
    }
    if (stamp) p.probe[c * 8 + 2] = rz::globaltimer_ns();
    prefetch(c + 2, cur);            // the loads of the chunk after next fly over one whole iteration
    rz::fence_proxy_async();
    if (stamp) p.probe[c * 8 + 3] = rz::globaltimer_ns();
    rz::tc_fence_before();
    __syncthreads();
    if (stamp) p.probe[c * 8 + 4] = rz::globaltimer_ns();
    if (tid == 0) {
      rz::tc_fence_after();
      rz::mbar_wait(bar_w + 8 * s, (uint32_t)(c / p.n_wslots) & 1u);
      if (stamp) p.probe[c * 8 + 5] = rz::globaltimer_ns();
      const uint64_t d_ahi = rz::umma_desc_sw128(a_hi), d_alo = rz::umma_desc_sw128(a_lo);
      if (policy) {
        // N = AS in pieces of at most 256 columns (AS = 384 for 19x19 Go: 256 + 128)
        for (int n0 = 0; n0 < AS; n0 += 256) {
          const int nn = min(256, AS - n0);
          const uint32_t idesc = rz::umma_idesc_bf16(128, nn);
          const uint64_t d_whi = rz::umma_desc_sw128(w_hi + (uint32_t)n0 * 128u);
          const uint64_t d_wlo = rz::umma_desc_sw128(w_lo + (uint32_t)n0 * 128u);
          const uint32_t d = tmem_base + (uint32_t)n0;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            rz::umma_bf16(d, d_ahi + (uint64_t)(2 * kk), d_whi + (uint64_t)(2 * kk), idesc, (c > 0 || kk > 0) ? 1u : 0u);
            rz::umma_bf16(d, d_alo + (uint64_t)(2 * kk), d_whi + (uint64_t)(2 * kk), idesc, 1u);
            rz::umma_bf16(d, d_ahi + (uint64_t)(2 * kk), d_wlo + (uint64_t)(2 * kk), idesc, 1u);
          }
        }
      } else {
        const uint64_t d_whi = rz::umma_desc_sw128(w_hi), d_wlo = rz::umma_desc_sw128(w_lo);
        const uint32_t d = tmem_base + (uint32_t)AS;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          rz::umma_bf16(d, d_ahi + (uint64_t)(2 * kk), d_whi + (uint64_t)(2 * kk), idesc_v, (c > n_pol || kk > 0) ? 1u : 0u);
          rz::umma_bf16(d, d_alo + (uint64_t)(2 * kk), d_whi + (uint64_t)(2 * kk), idesc_v, 1u);
          rz::umma_bf16(d, d_ahi + (uint64_t)(2 * kk), d_wlo + (uint64_t)(2 * kk), idesc_v, 1u);
        }
      }
      rz::umma_commit(bar_afree);
      if (c == n_chunks - 1) rz::umma_commit(bar_done);
      if (stamp) p.probe[c * 8 + 6] = rz::globaltimer_ns();
    }
  };
  for (int c = 0; c < n_chunks; c += 2) {
    step(c, pre[0]);
    if (c + 1 < n_chunks) step(c + 1, pre[1]);
  }
  rz::mbar_wait(bar_done, 0);
  rz::tc_fence_after();

  // ---- epilogue: warps 0..3 = log_softmax of board row (warp*32 + lane); warps 4..7 = the value of the same rows
  const int q = warp & 3;
  const int row = q * 32 + lane;
  const bool live = b0 + row < p.n_boards;
  const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
  if (warp < 4) {
    // act_fc1 bias + log_softmax over the A real outputs (:43-44); three sweeps over the TMEM row
    float mx = -3.0e38f;
    for (int c0 = 0; c0 < AS; c0 += 32) {
      uint32_t acc[32];
      rz::tmem_ld_32x32(t_row + (uint32_t)c0, acc);
      rz::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (c0 + j < p.A) mx = fmaxf(mx, __uint_as_float(acc[j]) + s_bp[c0 + j]);
    }
    float sum = 0.0f;
    for (int c0 = 0; c0 < AS; c0 += 32) {
      uint32_t acc[32];
      rz::tmem_ld_32x32(t_row + (uint32_t)c0, acc);
      rz::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (c0 + j < p.A) sum += expf((__uint_as_float(acc[j]) + s_bp[c0 + j]) - mx);
    }
    const float lse = mx + logf(sum);
    float* lp = p.logp + (size_t)(b0 + row) * AS;
    for (int c0 = 0; c0 < AS; c0 += 32) {
      uint32_t acc[32];
      rz::tmem_ld_32x32(t_row + (uint32_t)c0, acc);
      rz::tmem_ld_wait();
      if (live) {
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8) {
          uint32_t o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int j = j8 * 8 + e;
            o[e] = c0 + j < p.A ? __float_as_uint((__uint_as_float(acc[j]) + s_bp[c0 + j]) - lse) : 0u;
          }
          rz::st_global_v8(lp + c0 + j8 * 8, o);
        }
      }
    }
  } else {
    // val_fc1 bias + ReLU, val_fc2, tanh (:49-51)
    float hv = 0.0f;
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 32) {
      uint32_t acc[32];
      rz::tmem_ld_32x32(t_row + (uint32_t)(AS + c0), acc);
      rz::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j)
        hv = fmaf(fmaxf(__uint_as_float(acc[j]) + s_bv1[c0 + j], 0.0f), s_wv2[c0 + j], hv);
    }
    if (live) p.value[b0 + row] = tanhf(hv + p.bv2[0]);
  }
  rz::tc_fence_before();
  __syncthreads();
  if (warp == 0) { rz::tc_fence_after(); rz::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols); }
}


// ---- the same GEMM split over K across a cluster of four CTAs (action_stride <= 256) -------------------------------------
// One CTA streams 1.2 MB of split weights and converts 6P features per board chunk after chunk: 55 us for a single board,
// 84 us for 8192 (64 CTAs on 148 SMs) -- profiles/r2_run38_*, run40.  Here the HT4_CLUSTER = 4 CTAs of a cluster share the 128 boards
// of a tile: CTA r takes the feature chunks r, r + 4, r + 8, ... (its own share of the weights and of the conversion
// work), accumulates a partial [128 boards][AS + 64] product in its TMEM, and the partials meet through
// distributed shared memory: the rows of boards 32 r .. 32 r + 31 of every CTA's accumulator go to CTA r, which adds the
// partials in rank order and finishes log_softmax / the value head for its boards.  The arithmetic of a board does
// not depend on how many boards are evaluated, nor on its place in the tile.
constexpr int HT4_CLUSTER = 4;                  // CTAs per 128-board tile.  (8 was measured: 18 instead of 20 us for one board,
                                                // but 150 instead of 76 us for 8192 -- clusters of eight 199 KB CTAs schedule badly;
                                                // profiles/r2_run55_*.  The size is fixed: it defines the summation order.)
constexpr int HT4_ROWS = 128 / HT4_CLUSTER;     // boards a CTA finishes
constexpr int HT4_RSTRIDE = HT4_ROWS + 1;       // floats per column of the exchange buffers (+ 1: no bank conflicts)

__device__ __forceinline__ void st_cluster_f32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.b32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}

__global__ void __launch_bounds__(HT_THREADS, 1)
rz_heads_tc4_kernel(const __grid_constant__ CUtensorMap tmap_whi, const __grid_constant__ CUtensorMap tmap_wlo,
                    const __grid_constant__ CUtensorMap tmap_vhi, const __grid_constant__ CUtensorMap tmap_vlo,
                    const HeadsTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = rz::smem_u32(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int AS = p.AS, P = p.P, NC = p.AS + 64;
  const uint32_t rank = rz::cluster_ctarank();
  const uint32_t stage_bytes = 2u * HT_A_BYTES + ht_slot_bytes(AS);       // A_hi | A_lo | W_hi | W_lo
  const uint32_t ctrl = base + 2u * stage_bytes;
  uint8_t* ctrl_ptr = smem_raw + 2u * stage_bytes;
  const uint32_t bar_w = ctrl, bar_free = ctrl + 16, bar_done = ctrl + 32;   // [2], [2], [1]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ctrl_ptr + 48);
  float* s_bp = reinterpret_cast<float*>(ctrl_ptr + 64);        // [AS <= 256]
  float* s_bv1 = s_bp + 384;                                    // [64]
  float* s_wv2 = s_bv1 + 64;                                    // [64]

  const int b0 = (blockIdx.x / HT4_CLUSTER) * 128;
  const int r = tid & 127, khalf = tid >> 7;          // this thread builds row r, k in [32*khalf, 32*khalf + 32)
  const bool row_live = b0 + r < p.n_boards;
  const int K6 = 6 * P, K4 = 4 * P;
  // Chunks that hold only padding squares are skipped: a plane of the padded layout is P = S*S features of which the
  // first H*S are rows of the board (their zero features times zero weights add exact zeros, so the result is the
  // same bit for bit): 6 of 24 chunks for a 3x3 board at stride 16, 12 for 6x6, all 24 for 15x15.  The LIVE chunks,
  // numbered j = 0, 1, ... in ascending k, go round robin over the CTAs: CTA r takes j = r, r + 4, ...
  const int cpp = P >> 6, lpp = p.live_per_plane;               // chunks per plane: all, live
  const int n_live = 6 * lpp, n_pol_live = 4 * lpp;
  auto chunk_of = [&](int j) { return (j / lpp) * cpp + (j % lpp); };
  const int n_my = (n_live - (int)rank + HT4_CLUSTER - 1) / HT4_CLUSTER;
  const bool has_pol = (int)rank < n_pol_live;
  const int first_val_j = (int)rank + (((int)rank < n_pol_live) ? (n_pol_live - (int)rank + HT4_CLUSTER - 1) / HT4_CLUSTER * HT4_CLUSTER : 0);
  const bool has_val = first_val_j < n_live;
  const int n_pol = K4 >> 6;

  auto issue_w = [&](int i) {                         // weights of own chunk i into stage i & 1 (thread 0)
    const int c = chunk_of((int)rank + HT4_CLUSTER * i), s = i & 1;
    const uint32_t w_hi = base + (uint32_t)s * stage_bytes + 2 * HT_A_BYTES, w_lo = w_hi + ht_w_rows(AS) * 128u;
    if (c < n_pol) {
      rz::mbar_expect_tx(bar_w + 8 * s, 2u * (uint32_t)AS * 128u);
      for (int j = 0; j < AS; j += p.w_box) {
        rz::tma_load_2d(w_hi + (uint32_t)j * 128u, &tmap_whi, bar_w + 8 * s, c * 64, j);
        rz::tma_load_2d(w_lo + (uint32_t)j * 128u, &tmap_wlo, bar_w + 8 * s, c * 64, j);
      }
    } else {
      rz::mbar_expect_tx(bar_w + 8 * s, 2u * 64u * 128u);
      rz::tma_load_2d(w_hi, &tmap_vhi, bar_w + 8 * s, c * 64, 0);
      rz::tma_load_2d(w_lo, &tmap_vlo, bar_w + 8 * s, c * 64, 0);
    }
  };

  if (tid == 0) {
    if (base & 1023u) __trap();
    rz::tma_prefetch_desc(&tmap_whi);
    rz::tma_prefetch_desc(&tmap_wlo);
    rz::tma_prefetch_desc(&tmap_vhi);
    rz::tma_prefetch_desc(&tmap_vlo);
    for (int s = 0; s < 2; ++s) { rz::mbar_init(bar_w + 8 * s, 1); rz::mbar_init(bar_free + 8 * s, 1); }
    rz::mbar_init(bar_done, 1);
    rz::fence_barrier_init();
    // static weights: the first two chunks are requested before the grid dependency resolves
    for (int i = 0; i < 2 && i < n_my; ++i) issue_w(i);
  }
  if (warp == 0) { rz::tmem_alloc(rz::smem_u32(tmem_holder), (uint32_t)p.tmem_cols); rz::tmem_relinquish(); }
  for (int i = tid; i < AS; i += HT_THREADS) s_bp[i] = i < p.A ? p.bp[i] : 0.0f;
  if (tid < 64) { s_bv1[tid] = p.bv1[tid]; s_wv2[tid] = p.wv2[tid]; }
  rz::grid_dep_wait();     // programmatic dependent launch (rz_common.cuh): the features come from the previous kernel
  rz::grid_dep_launch();
  rz::tc_fence_before();
  __syncthreads();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  const float* frow = p.feat + (size_t)(b0 + r) * K6 + 32 * khalf;
  float4 pre[2][8];                                   // the features of own chunks i, i + 1 in registers
  auto prefetch = [&](int i, float4 (&dst)[8]) {
    const int c = chunk_of((int)rank + HT4_CLUSTER * i);
    const int k0 = c * 64 + 32 * khalf;
    const bool live = row_live && i < n_my && k0 < K6;   // K6 is a multiple of 32
    const float4* src = reinterpret_cast<const float4*>(frow + (size_t)c * 64);
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[j] = live ? __ldg(src + j) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  };
  prefetch(0, pre[0]);
  prefetch(1, pre[1]);

  const uint32_t idesc_v = rz::umma_idesc_bf16(128, 64);
  const uint32_t idesc_p = rz::umma_idesc_bf16(128, AS);
  auto step = [&](const int i, float4 (&cur)[8]) {
    const int j_live = (int)rank + HT4_CLUSTER * i, c = chunk_of(j_live), s = i & 1;
    const uint32_t st = base + (uint32_t)s * stage_bytes;
    const uint32_t a_hi = st, a_lo = st + HT_A_BYTES, w_hi = st + 2 * HT_A_BYTES, w_lo = w_hi + ht_w_rows(AS) * 128u;
    const bool policy = c < n_pol;
    if (i >= 2) rz::mbar_wait(bar_free + 8 * s, (uint32_t)((i >> 1) - 1) & 1u);   // MMAs of own chunk i - 2 have read the stage
    {
      const uint32_t row_off = (uint32_t)r * 128u;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float x[8] = {cur[2 * q].x, cur[2 * q].y, cur[2 * q].z, cur[2 * q].w,
                            cur[2 * q + 1].x, cur[2 * q + 1].y, cur[2 * q + 1].z, cur[2 * q + 1].w};
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * e]), h1 = __float2bfloat16_rn(x[2 * e + 1]);
          hi[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
          lo[e] = rz::pack_bf16x2(x[2 * e] - __bfloat162float(h0), x[2 * e + 1] - __bfloat162float(h1));
        }
        const uint32_t chunk = (uint32_t)(khalf * 4 + q);
        const uint32_t off = row_off + ((chunk ^ ((uint32_t)r & 7u)) << 4);
        rz::st_shared_v4(a_hi + off, hi[0], hi[1], hi[2], hi[3]);
        rz::st_shared_v4(a_lo + off, lo[0], lo[1], lo[2], lo[3]);
      }
    }
    prefetch(i + 2, cur);
    rz::fence_proxy_async();
    rz::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      rz::tc_fence_after();
      rz::mbar_wait(bar_w + 8 * s, (uint32_t)(i >> 1) & 1u);
      const uint64_t d_ahi = rz::umma_desc_sw128(a_hi), d_alo = rz::umma_desc_sw128(a_lo);
      const uint64_t d_whi = rz::umma_desc_sw128(w_hi), d_wlo = rz::umma_desc_sw128(w_lo);
      const uint32_t d = tmem_base + (policy ? 0u : (uint32_t)AS);
      const uint32_t idesc = policy ? idesc_p : idesc_v;
      const bool first = policy ? (i == 0) : (j_live == first_val_j);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        rz::umma_bf16(d, d_ahi + (uint64_t)(2 * kk), d_whi + (uint64_t)(2 * kk), idesc, (!first || kk > 0) ? 1u : 0u);
        rz::umma_bf16(d, d_alo + (uint64_t)(2 * kk), d_whi + (uint64_t)(2 * kk), idesc, 1u);
        rz::umma_bf16(d, d_ahi + (uint64_t)(2 * kk), d_wlo + (uint64_t)(2 * kk), idesc, 1u);
      }
      rz::umma_commit(bar_free + 8 * s);
      if (i == n_my - 1) rz::umma_commit(bar_done);
      // the other stage's weights for own chunk i + 1 were requested after chunk i - 1; now those of chunk i + 2 can
      // follow chunk i into this stage as soon as its MMAs are done -- requested after the NEXT chunk's MMAs are issued
      if (i >= 1 && i + 1 < n_my) {
        rz::mbar_wait(bar_free + 8 * (s ^ 1), (uint32_t)(((i - 1) >> 1)) & 1u);   // MMAs of own chunk i - 1 done
        issue_w(i + 1);
      }
    }
  };
  for (int i = 0; i < n_my; i += 2) {
    step(i, pre[0]);
    if (i + 1 < n_my) step(i + 1, pre[1]);
  }
  if (n_my > 0) rz::mbar_wait(bar_done, 0);
  rz::tc_fence_after();

  // ---- exchange: every CTA has finished its MMAs, the stages are dead: they become the receive buffers
  // rb[src rank][column][HT4_RSTRIDE] float32 of the HT4_ROWS boards this CTA finishes
  rz::cluster_sync_all();
  const uint32_t rb = base;
  {
    const int q = warp & 3;                                     // TMEM lane quarter = destination CTA
    const int ng = NC >> 5, g0 = (warp >> 2) ? (ng + 1) / 2 : 0, g1 = (warp >> 2) ? ng : (ng + 1) / 2;
    const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
    for (int g = g0; g < g1; ++g) {
      const int c0 = g * 32;
      uint32_t acc[32];
      const bool has = c0 < AS ? has_pol : has_val;
      if (has) { rz::tmem_ld_32x32(t_row + (uint32_t)c0, acc); rz::tmem_ld_wait(); }
      else {
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = 0u;
      }
      // board row q * 32 + lane of the tile is finished by CTA (q * 32 + lane) / HT4_ROWS, as its row (lane % HT4_ROWS)
      const uint32_t dst = rz::mapa_shared(rb + (uint32_t)((((int)rank * NC + c0) * HT4_RSTRIDE + (lane % HT4_ROWS)) * 4),
                                           (uint32_t)((q * 32 + lane) / HT4_ROWS));
#pragma unroll
      for (int j = 0; j < 32; ++j) st_cluster_f32(dst + (uint32_t)(j * HT4_RSTRIDE * 4), acc[j]);
    }
  }
  rz::tc_fence_before();
  rz::cluster_sync_all();

  // ---- finish boards b0 + 32 rank + (0..31): partials added in rank order, biases, log_softmax / value head
  float* rbf = reinterpret_cast<float*>(smem_raw);
  for (int idx = tid; idx < NC * HT4_ROWS; idx += HT_THREADS) {
    const int col = idx / HT4_ROWS, row = idx % HT4_ROWS;
    const int o = col * HT4_RSTRIDE + row;
    float v = rbf[o];
#pragma unroll
    for (int src = 1; src < HT4_CLUSTER; ++src) v += rbf[src * NC * HT4_RSTRIDE + o];
    rbf[o] = v + (col < AS ? s_bp[col] : s_bv1[col - AS]);
  }
  __syncthreads();
  for (int rr = warp; rr < HT4_ROWS; rr += HT_THREADS / 32) {     // one warp per board
    const int board = b0 + HT4_ROWS * (int)rank + rr;
    // act_fc1 + log_softmax over the A real outputs (:43-44): lanes stride over the columns, butterfly reductions
    float mx = -3.0e38f;
    for (int c = lane; c < p.A; c += 32) mx = fmaxf(mx, rbf[c * HT4_RSTRIDE + rr]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(RZ_FULL, mx, o));
    float sum = 0.0f;
    for (int c = lane; c < p.A; c += 32) sum += expf(rbf[c * HT4_RSTRIDE + rr] - mx);
    sum = rz_warp_sum_f32(sum);
    const float lse = mx + logf(sum);
    // val_fc1 + ReLU, val_fc2, tanh (:49-51)
    float hv = fmaf(fmaxf(rbf[(AS + lane) * HT4_RSTRIDE + rr], 0.0f), s_wv2[lane],
                    fmaxf(rbf[(AS + 32 + lane) * HT4_RSTRIDE + rr], 0.0f) * s_wv2[32 + lane]);
    hv = rz_warp_sum_f32(hv);
    if (board < p.n_boards) {
      float* lp = p.logp + (size_t)board * AS;
      for (int c = lane; c < AS; c += 32) lp[c] = c < p.A ? rbf[c * HT4_RSTRIDE + rr] - lse : 0.0f;
      if (lane == 0) p.value[board] = tanhf(hv + p.bv2[0]);
    }
  }
  rz::tc_fence_before();
  __syncthreads();
  if (warp == 0) { rz::tc_fence_after(); rz::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols); }
}

}  // namespace

extern "C" int rz_net_heads_tc(const rz_heads_desc* h, const float* feat, float* logp, float* value,
                               int n_boards, void* stream) {
  RZ_REQUIRE(h && feat && logp && value, "rz_net_heads_tc: null argument");
  RZ_REQUIRE(h->wtc_hi && h->wtc_lo && h->bp && h->bv1 && h->wv2 && h->bv2, "rz_net_heads_tc: null weight pointer");
  RZ_REQUIRE(h->board_size >= 1 && h->board_size <= RZ_MAX_BOARD, "rz_net_heads_tc: board_size %d", h->board_size);
  const int W = h->width > 0 ? h->width : h->board_size;
  RZ_REQUIRE(W >= 1 && W <= RZ_MAX_BOARD, "rz_net_heads_tc: width %d", W);
  const int A = h->n_actions > 0 ? h->n_actions : h->board_size * W;
  const int AS = h->action_stride;
  RZ_REQUIRE(AS >= A && (AS & 31) == 0 && AS <= 384, "rz_net_heads_tc: action_stride %d", AS);
  const int S = rz_row_stride(h->board_size, W, h->row_stride);
  RZ_REQUIRE(S != 0, "rz_net_heads_tc: row_stride %d does not hold a %dx%d board", h->row_stride, h->board_size, W);
  RZ_REQUIRE(n_boards >= 0, "rz_net_heads_tc: n_boards %d", n_boards);
  if (n_boards == 0) return 0;
  const int P = S * S;
  const int KP = (6 * P + 63) / 64 * 64;
  HeadsTcParams p;
  p.feat = feat; p.bp = h->bp; p.bv1 = h->bv1; p.wv2 = h->wv2; p.bv2 = h->bv2; p.logp = logp; p.value = value;
  p.n_boards = n_boards; p.A = A; p.AS = AS; p.P = P;
  p.probe = rz_probe_buffer;
  // rows 0 .. H-1 of a plane are real squares: ceil(H*S / 64) of its P / 64 chunks (P is 64 or 256 in the cluster kernel)
  p.live_per_plane = (P % 64 == 0) ? ((h->board_size * S + 63) / 64 < P / 64 ? (h->board_size * S + 63) / 64 : P / 64) : 0;
  p.w_box = (AS % 128 == 0) ? 128 : ((AS % 64 == 0) ? 64 : 32);
  p.tmem_cols = 32;
  while (p.tmem_cols < AS + 64) p.tmem_cols *= 2;
  const size_t slot = ht_slot_bytes(AS);
  p.n_wslots = (int)((232448 - HT_CTRL_BYTES - 2 * HT_A_BYTES) / slot);
  if (p.n_wslots > 4) p.n_wslots = 4;
  RZ_REQUIRE(p.n_wslots >= 2, "rz_net_heads_tc: action_stride %d leaves room for %d weight slots", AS, p.n_wslots);
  const size_t smem = 2 * HT_A_BYTES + (size_t)p.n_wslots * slot + HT_CTRL_BYTES;
  // weights: bf16 [AS + 64][KP] K-major, rows 0..AS-1 the policy outputs, AS..AS+63 the value hidden units
  const __nv_bfloat16* whi = reinterpret_cast<const __nv_bfloat16*>(h->wtc_hi);
  const __nv_bfloat16* wlo = reinterpret_cast<const __nv_bfloat16*>(h->wtc_lo);
  CUtensorMap t_whi, t_wlo, t_vhi, t_vlo;
  if (rz::make_tmap_2d(&t_whi, whi, (uint64_t)AS, (uint64_t)KP, (uint32_t)p.w_box)) return -1;
  if (rz::make_tmap_2d(&t_wlo, wlo, (uint64_t)AS, (uint64_t)KP, (uint32_t)p.w_box)) return -1;
  if (rz::make_tmap_2d(&t_vhi, whi + (size_t)AS * KP, 64, (uint64_t)KP, 64)) return -1;
  if (rz::make_tmap_2d(&t_vlo, wlo + (size_t)AS * KP, 64, (uint64_t)KP, 64)) return -1;
  if (AS <= 256 && p.live_per_plane > 0) {
    // the cluster-of-four split-K kernel
    const size_t smem4 = 2 * (2 * HT_A_BYTES + slot) + HT_CTRL_BYTES;
    static size_t attr_smem4 = 0;
    if (smem4 > attr_smem4) {
      cudaError_t e = cudaFuncSetAttribute(rz_heads_tc4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4);
      if (e != cudaSuccess) { rz_set_error("rz_net_heads_tc: smem attribute: %s", cudaGetErrorString(e)); return -2; }
      attr_smem4 = smem4;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(HT4_CLUSTER * ((n_boards + 127) / 128)));
    cfg.blockDim = dim3(HT_THREADS);
    cfg.dynamicSmemBytes = smem4;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = HT4_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1 + rz_pdl_attr(&attr[1]);
    cudaError_t e = cudaLaunchKernelEx(&cfg, rz_heads_tc4_kernel, t_whi, t_wlo, t_vhi, t_vlo, p);
    if (e != cudaSuccess) { rz_set_error("rz_net_heads_tc: launch failed: %s", cudaGetErrorString(e)); return -2; }
    return 0;
  }
  static size_t attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(rz_heads_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { rz_set_error("rz_net_heads_tc: smem attribute: %s", cudaGetErrorString(e)); return -2; }
    attr_smem = smem;
  }
  const int grid = (n_boards + 127) / 128;
  rz_launch_pdl(rz_heads_tc_kernel, grid, HT_THREADS, smem, (cudaStream_t)stream, t_whi, t_wlo, t_vhi, t_vlo, p);
  RZ_LAUNCH_CHECK("rz_net_heads_tc");
  return 0;
}
