// rlzero_b200 -- policy / value heads and the generic fp32 3x3 convolution.
//
// Reference: rlzero/games/gomoku/policy_value_net.py
//   trunk  conv1..3 (3x3, pad 1) + ReLU                         :14-16, 36-38
//   policy act_conv1 (1x1 -> 4) + ReLU, act_fc1 (4HW -> HW), log_softmax   :19-21, 41-44
//   value  val_conv1 (1x1 -> 2) + ReLU, val_fc1 (2HW -> 64) + ReLU, val_fc2 (64 -> 1), tanh  :23-25, 47-51
// The flatten order of x.view(-1, C*H*W) on an NCHW tensor is c*HW + pos; the fully connected
// weights are stored transposed ([in][out]) so that threads over `out` read them coalesced.
//
// The fp32 convolution is the plain CUDA-core path used for the reference's stock network
// (3 layers, <= 64 input channels) at any board size, and the heads kernel finishes it.  The
// tensor-core trunks end in rz_net_heads_tc.cu, fed by the head-features kernel below.
#include <cuda_bf16.h>
#include <string.h>

#include "rz_common.cuh"

namespace {

// ---------------------------------------------------------------------------
// fp32 conv3x3, NHWC: in [B][HW][Cin], w [9][Cin][Cout], out [B][HW][Cout]
// blockIdx.x = board, blockIdx.y = slice of the board's (position, output channel) pairs: a single game (the
// reference API, batch 1) is spread over gridDim.y blocks instead of one SM; the input board sits in shared memory.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rz_conv3x3_f32_kernel(const float* __restrict__ in, const float* __restrict__ w,
                      const float* __restrict__ bias, const float* __restrict__ residual,
                      float* __restrict__ out, int H, int Cin, int Cout, int relu) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  extern __shared__ float s_in[];  // [HW][Cin]
  const int b = blockIdx.x, HW = H * H;
  const float* ib = in + (size_t)b * HW * Cin;
  for (int i = threadIdx.x; i < HW * Cin; i += blockDim.x) s_in[i] = ib[i];
  __syncthreads();
  const int total = HW * Cout;
  const int per = (total + gridDim.y - 1) / gridDim.y;
  const int lo = blockIdx.y * per, hi = min(total, lo + per);
  for (int idx = lo + threadIdx.x; idx < hi; idx += blockDim.x) {
    const int co = idx % Cout, pos = idx / Cout;
    const int y = pos / H, x = pos - y * H;
    float acc = bias[co];
    for (int tap = 0; tap < 9; ++tap) {
      const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
      if (yy < 0 || yy >= H || xx < 0 || xx >= H) continue;
      const float* src = s_in + (yy * H + xx) * Cin;
      const float* wt = w + (size_t)tap * Cin * Cout + co;
      for (int ci = 0; ci < Cin; ++ci) acc = fmaf(src[ci], wt[(size_t)ci * Cout], acc);
    }
    const size_t o = ((size_t)b * HW + pos) * Cout + co;
    if (residual) acc += residual[o];
    if (relu) acc = fmaxf(acc, 0.0f);
    out[o] = acc;
  }
}

// The same operator register-tiled: a thread owns TP consecutive positions x 4 consecutive output channels, so one
// 128-bit weight load and TP shared-memory reads feed 4*TP FMAs (the kernel above issues two loads per FMA).  Every
// output accumulates bias, then taps 0..8 (in-board only), input channels ascending, with the same fmaf operand order
// as above: the results are bit-identical to it (tests compare the fp32 path with live-reference fixtures).
template <int TP>
__global__ void __launch_bounds__(256)
rz_conv3x3_f32_tiled_kernel(const float* __restrict__ in, const float* __restrict__ w,
                            const float* __restrict__ bias, const float* __restrict__ residual,
                            float* __restrict__ out, int H, int Cin, int Cout, int relu) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  extern __shared__ float s_in[];  // [HW][Cin]
  const int b = blockIdx.x, HW = H * H;
  const float* ib = in + (size_t)b * HW * Cin;
  for (int i = threadIdx.x; i < HW * Cin; i += blockDim.x) s_in[i] = ib[i];
  __syncthreads();
  const int ct = Cout >> 2, pt = (HW + TP - 1) / TP;
  const int total = ct * pt;
  const int per = (total + gridDim.y - 1) / gridDim.y;
  const int lo = blockIdx.y * per, hi = min(total, lo + per);
  for (int t = lo + threadIdx.x; t < hi; t += blockDim.x) {
    const int co0 = (t % ct) << 2, pos0 = (t / ct) * TP;
    const float4 b4 = *reinterpret_cast<const float4*>(bias + co0);
    float acc[TP][4];
    int py[TP], px[TP];
#pragma unroll
    for (int p = 0; p < TP; ++p) {
      acc[p][0] = b4.x; acc[p][1] = b4.y; acc[p][2] = b4.z; acc[p][3] = b4.w;
      const int pos = pos0 + p;
      py[p] = pos < HW ? pos / H : -4;          // -4: every tap of a position beyond the board is out of range
      px[p] = pos - (pos / H) * H;
    }
    for (int tap = 0; tap < 9; ++tap) {
      const int dy = tap / 3 - 1, dx = tap % 3 - 1;
      int base[TP];
      bool ok[TP], any = false;
#pragma unroll
      for (int p = 0; p < TP; ++p) {
        const int yy = py[p] + dy, xx = px[p] + dx;
        ok[p] = yy >= 0 && yy < H && xx >= 0 && xx < H;
        base[p] = ok[p] ? (yy * H + xx) * Cin : 0;
        any |= ok[p];
      }
      if (!any) continue;
      const float* wt = w + (size_t)tap * Cin * Cout + co0;
      for (int ci = 0; ci < Cin; ++ci) {
        const float4 w4 = *reinterpret_cast<const float4*>(wt + (size_t)ci * Cout);
#pragma unroll
        for (int p = 0; p < TP; ++p) {
          if (ok[p]) {
            const float x = s_in[base[p] + ci];
            acc[p][0] = fmaf(x, w4.x, acc[p][0]);
            acc[p][1] = fmaf(x, w4.y, acc[p][1]);
            acc[p][2] = fmaf(x, w4.z, acc[p][2]);
            acc[p][3] = fmaf(x, w4.w, acc[p][3]);
          }
        }
      }
    }
#pragma unroll
    for (int p = 0; p < TP; ++p) {
      const int pos = pos0 + p;
      if (pos >= HW) continue;
      const size_t o = ((size_t)b * HW + pos) * Cout + co0;
      float4 r = make_float4(acc[p][0], acc[p][1], acc[p][2], acc[p][3]);
      if (residual) {
        const float4 q = *reinterpret_cast<const float4*>(residual + o);
        r.x += q.x; r.y += q.y; r.z += q.z; r.w += q.w;
      }
      if (relu) { r.x = fmaxf(r.x, 0.0f); r.y = fmaxf(r.y, 0.0f); r.z = fmaxf(r.z, 0.0f); r.w = fmaxf(r.w, 0.0f); }
      *reinterpret_cast<float4*>(out + o) = r;
    }
  }
}

// ---------------------------------------------------------------------------
// heads: NB boards per block.
//
// Shared-memory feature layout is [k][NB] (k = flattened FC input index c*HW + pos, policy
// features first, value features after them), so that the FC loops read the NB boards of one k
// as float4 broadcasts: per k a thread issues 1 coalesced weight load + NB/4 LDS.128 + NB FMAs.
// (The first revision kept [board][k] and spent 54 M shared-memory wavefronts per launch on
// scalar broadcasts -- profiles/r1_run4_*: 532 us for 6.6 GFLOP.)
// ---------------------------------------------------------------------------
constexpr int HEAD_NB = 16;
constexpr int HEAD_THREADS = 256;
constexpr int HEAD_C = 128;

struct HeadsParams {
  const void* act;        // trunk output: fp32 [B][HW][128] (heads) or bf16 [B*P][128] (padded layout, features)
  const float* w1x1;      // [6][128]: 4 policy + 2 value 1x1 filters
  const float* b1x1;      // [6]
  const float* wp;        // [4*HW + 4][AS] policy FC, transposed + padded (4 zero rows at the end)
  const float* bp;        // [AS]
  const float* wv1;       // [2*HW + 2][64] value FC1, transposed (2 zero rows at the end)
  const float* bv1;       // [64]
  const float* wv2;       // [64]
  const float* bv2;       // [1]
  float* logp;            // [B][AS]
  float* value;           // [B]
  int n_boards, H, W, HW, A, AS;   // H x W squares (HW), A policy outputs
  int S, P;                        // padded layout of a bf16 source: row stride S, P = S*S rows per board
};

// 256-bit read-only global load: one full 32-byte sector per lane (sm_100 LDG.E.256)
__device__ __forceinline__ void rz_ld_global_nc_v8(const void* p, uint32_t (&r)[8]) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p));
}

// 6 dot products of one position's 128 channels with the 1x1 filters in shared memory.  Summation order
// (shared with the fused epilogue of rz_net_tc2.cu, which splits a row over two warps): channels 0..63
// ascending onto the bias, channels 64..127 ascending onto zero, then the two partial sums are added.
template <bool kTile>
__device__ __forceinline__ void conv1x1_position(const void* act, int b, int pos, int W, int HW, int S, int P,
                                                 const float* __restrict__ s_w, float (&acc)[6]) {
  const float4* w4 = reinterpret_cast<const float4*>(s_w);
  float hi[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
  if constexpr (kTile) {
    const int y = pos / W, x = pos - y * W;
    const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(act) + ((size_t)b * P + y * S + x) * HEAD_C;
    uint32_t raw[8][8];  // the whole row: 8 x 32 B, all loads in flight before the first use
#pragma unroll
    for (int j = 0; j < 8; ++j) rz_ld_global_nc_v8(src + j * 16, raw[j]);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      float v[8];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t q = raw[j >> 1][(j & 1) * 4 + e];
        v[2 * e] = __uint_as_float(q << 16);
        v[2 * e + 1] = __uint_as_float(q & 0xffff0000u);
      }
#pragma unroll
      for (int f = 0; f < 6; ++f) {
        const float4 wa = w4[f * (HEAD_C / 4) + j * 2], wb = w4[f * (HEAD_C / 4) + j * 2 + 1];
        float a = j < 8 ? acc[f] : hi[f];
        a = fmaf(v[0], wa.x, a); a = fmaf(v[1], wa.y, a); a = fmaf(v[2], wa.z, a); a = fmaf(v[3], wa.w, a);
        a = fmaf(v[4], wb.x, a); a = fmaf(v[5], wb.y, a); a = fmaf(v[6], wb.z, a); a = fmaf(v[7], wb.w, a);
        if (j < 8) acc[f] = a; else hi[f] = a;
      }
    }
  } else {
    const float4* src = reinterpret_cast<const float4*>(
        reinterpret_cast<const float*>(act) + ((size_t)b * HW + pos) * HEAD_C);
#pragma unroll 4
    for (int j = 0; j < HEAD_C / 4; ++j) {
      const float4 q = src[j];
#pragma unroll
      for (int f = 0; f < 6; ++f) {
        const float4 w = w4[f * (HEAD_C / 4) + j];
        float a = j < HEAD_C / 8 ? acc[f] : hi[f];
        a = fmaf(q.x, w.x, a); a = fmaf(q.y, w.y, a); a = fmaf(q.z, w.z, a); a = fmaf(q.w, w.w, a);
        if (j < HEAD_C / 8) acc[f] = a; else hi[f] = a;
      }
    }
  }
#pragma unroll
  for (int f = 0; f < 6; ++f) acc[f] += hi[f];
}

// feature (k, board bi) lives at s_f[k*NB + (((bi >> 2) ^ (k & 3)) << 2) + (bi & 3)]: the XOR keeps
// a float4 of 4 boards together (the FC loops read it as one broadcast LDS.128) while spreading
// writers that differ only in k over 8 banks
__device__ __forceinline__ int feat_slot(int k, int bi) {
  return k * HEAD_NB + ((((bi >> 2) ^ (k & 3)) << 2) | (bi & 3));
}

__global__ void __launch_bounds__(HEAD_THREADS, 2) rz_heads_kernel(const HeadsParams p) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  extern __shared__ __align__(16) float sm[];
  const int HW = p.HW;
  float* s_f = sm;                              // [6*HW][NB]  k-major features (policy 4*HW, then value 2*HW)
  float* s_lg = s_f + 6 * HW * HEAD_NB;         // [NB][AS]    logits
  float* s_h = s_lg + HEAD_NB * p.AS;           // [NB][64]    value hidden
  float* s_w = s_h + HEAD_NB * 64;              // [6][128]    1x1 filters
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b0 = blockIdx.x * HEAD_NB;
  const int nb = min(HEAD_NB, p.n_boards - b0);
  for (int i = tid; i < 6 * HEAD_C; i += HEAD_THREADS) s_w[i] = p.w1x1[i];
  __syncthreads();
  // phase 1: 1x1 convolutions + ReLU  (policy_value_net.py:41, 47); boards beyond nb hold zeros
  for (int i = tid; i < HEAD_NB * HW; i += HEAD_THREADS) {
    const int bi = i % HEAD_NB, pos = i / HEAD_NB;
    float acc[6];
#pragma unroll
    for (int f = 0; f < 6; ++f) acc[f] = p.b1x1[f];
    if (bi < nb) conv1x1_position<false>(p.act, b0 + bi, pos, p.W, HW, p.S, p.P, s_w, acc);
#pragma unroll
    for (int f = 0; f < 6; ++f) s_f[feat_slot(f * HW + pos, bi)] = bi < nb ? fmaxf(acc[f], 0.0f) : 0.0f;
  }
  __syncthreads();
  // phase 2: policy FC (:43).  Thread (half, t): output columns t and t+128 of every 256-column
  // group, for all NB boards, over one half of the k range: per k 2 coalesced weight loads
  // (prefetched 4 k ahead) + NB/4 broadcast LDS.128 feed 2*NB FMAs.
  {
    const int khalf = tid >> 7, t = tid & 127;
    // both halves of the k range are multiples of 4 (K = 4*HW); wp carries 4 zero rows of padding
    // after row K-1, so the prefetch never needs a bounds check
    const int K = 4 * HW, k_mid = (K >> 1) & ~3;
    const int k_lo = khalf ? k_mid : 0, k_hi = khalf ? K : k_mid;
    const float4* f4 = reinterpret_cast<const float4*>(s_f);
    for (int jb = 0; jb < p.AS; jb += 256) {
      const int j0 = jb + t, j1 = jb + 128 + t;
      const bool c0 = j0 < p.A, c1 = j1 < p.A;
      float acc0[HEAD_NB], acc1[HEAD_NB];
#pragma unroll
      for (int bi = 0; bi < HEAD_NB; ++bi) { acc0[bi] = 0.0f; acc1[bi] = 0.0f; }
      constexpr int PF = 4;
      const float* w0p = p.wp + (size_t)k_lo * p.AS + (c0 ? j0 : 0);
      const float* w1p = p.wp + (size_t)k_lo * p.AS + (c1 ? j1 : 0);
      const size_t step = (size_t)p.AS;
      float wn0[PF], wn1[PF];
#pragma unroll
      for (int u = 0; u < PF; ++u) { wn0[u] = w0p[u * step]; wn1[u] = w1p[u * step]; }
      for (int k = k_lo; k < k_hi; k += PF) {
        float w0[PF], w1[PF];
        w0p += PF * step;
        w1p += PF * step;
#pragma unroll
        for (int u = 0; u < PF; ++u) {
          w0[u] = wn0[u]; w1[u] = wn1[u];
          wn0[u] = w0p[u * step];
          wn1[u] = w1p[u * step];
        }
        const float4* fk = f4 + k * (HEAD_NB / 4);
#pragma unroll
        for (int u = 0; u < PF; ++u) {
#pragma unroll
          for (int g = 0; g < HEAD_NB / 4; ++g) {
            const float4 f = fk[u * (HEAD_NB / 4) + (g ^ u)];   // k is a multiple of 4: (k+u) & 3 == u
            acc0[g * 4 + 0] = fmaf(f.x, w0[u], acc0[g * 4 + 0]);
            acc0[g * 4 + 1] = fmaf(f.y, w0[u], acc0[g * 4 + 1]);
            acc0[g * 4 + 2] = fmaf(f.z, w0[u], acc0[g * 4 + 2]);
            acc0[g * 4 + 3] = fmaf(f.w, w0[u], acc0[g * 4 + 3]);
            acc1[g * 4 + 0] = fmaf(f.x, w1[u], acc1[g * 4 + 0]);
            acc1[g * 4 + 1] = fmaf(f.y, w1[u], acc1[g * 4 + 1]);
            acc1[g * 4 + 2] = fmaf(f.z, w1[u], acc1[g * 4 + 2]);
            acc1[g * 4 + 3] = fmaf(f.w, w1[u], acc1[g * 4 + 3]);
          }
        }
      }
      // the upper k half parks its partial sums in s_lg, the lower half adds its own + the bias
      if (khalf) {
#pragma unroll
        for (int bi = 0; bi < HEAD_NB; ++bi) {
          if (j0 < p.AS) s_lg[bi * p.AS + j0] = acc0[bi];
          if (j1 < p.AS) s_lg[bi * p.AS + j1] = acc1[bi];
        }
      }
      __syncthreads();
      if (!khalf) {
        const float bj0 = c0 ? p.bp[j0] : 0.0f, bj1 = c1 ? p.bp[j1] : 0.0f;
#pragma unroll
        for (int bi = 0; bi < HEAD_NB; ++bi) {
          if (j0 < p.AS) s_lg[bi * p.AS + j0] = c0 ? (acc0[bi] + s_lg[bi * p.AS + j0]) + bj0 : 0.0f;
          if (j1 < p.AS) s_lg[bi * p.AS + j1] = c1 ? (acc1[bi] + s_lg[bi * p.AS + j1]) + bj1 : 0.0f;
        }
      }
    }
  }
  // phase 3a: value FC1 + ReLU (:49): thread = (output o, group of 4 boards)
  for (int i = tid; i < (HEAD_NB / 4) * 64; i += HEAD_THREADS) {
    const int o = i & 63, g = i >> 6;
    const float bo = p.bv1[o];
    float a0 = bo, a1 = bo, a2 = bo, a3 = bo;
    const float4* f4 = reinterpret_cast<const float4*>(s_f + (size_t)4 * HW * HEAD_NB);
    // K = 2*HW is even and the value features start at k = 4*HW (a multiple of 4): unroll by 2,
    // swizzle phase (4*HW + k) & 3 = k & 3; wv1 carries 2 zero rows of padding for the prefetch
    const int K = 2 * HW;
    const float* wp1 = p.wv1 + o;
    float wn0 = wp1[0], wn1 = wp1[64];
    for (int k = 0; k < K; k += 2) {
      const float w0 = wn0, w1 = wn1;
      wp1 += 128;
      wn0 = wp1[0]; wn1 = wp1[64];
      const float4 fa = f4[k * (HEAD_NB / 4) + (g ^ (k & 3))];
      const float4 fb = f4[(k + 1) * (HEAD_NB / 4) + (g ^ ((k + 1) & 3))];
      a0 = fmaf(fa.x, w0, a0); a1 = fmaf(fa.y, w0, a1); a2 = fmaf(fa.z, w0, a2); a3 = fmaf(fa.w, w0, a3);
      a0 = fmaf(fb.x, w1, a0); a1 = fmaf(fb.y, w1, a1); a2 = fmaf(fb.z, w1, a2); a3 = fmaf(fb.w, w1, a3);
    }
    s_h[(g * 4 + 0) * 64 + o] = fmaxf(a0, 0.0f);
    s_h[(g * 4 + 1) * 64 + o] = fmaxf(a1, 0.0f);
    s_h[(g * 4 + 2) * 64 + o] = fmaxf(a2, 0.0f);
    s_h[(g * 4 + 3) * 64 + o] = fmaxf(a3, 0.0f);
  }
  __syncthreads();
  // phase 3b: log_softmax (:44) and value FC2 + tanh (:50-51): one warp per board
  for (int bi = warp; bi < nb; bi += HEAD_THREADS / 32) {
    float mx = -3.0e38f;
    for (int j = lane; j < p.A; j += 32) mx = fmaxf(mx, s_lg[bi * p.AS + j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(RZ_FULL, mx, o));
    float sum = 0.0f;
    for (int j = lane; j < p.A; j += 32) sum += expf(s_lg[bi * p.AS + j] - mx);
    sum = rz_warp_sum_f32(sum);
    const float lse = mx + logf(sum);
    float* lp = p.logp + (size_t)(b0 + bi) * p.AS;
    for (int j = lane; j < p.AS; j += 32) lp[j] = j < p.A ? s_lg[bi * p.AS + j] - lse : 0.0f;
    float hv = s_h[bi * 64 + lane] * p.wv2[lane] + s_h[bi * 64 + 32 + lane] * p.wv2[32 + lane];
    hv = rz_warp_sum_f32(hv);
    if (lane == 0) p.value[b0 + bi] = tanhf(hv + p.bv2[0]);
  }
}

// the heads' 1x1 convolutions + ReLU alone: bf16 trunk output (padded layout) -> feat[b][f][y*S+x], the tensor the
// fused last trunk layer writes from its epilogue (same summation order, conv1x1_position).  Padding squares hold
// relu(bias), as there (their activations are zero); the FC weights are zero at those columns.
__global__ void __launch_bounds__(256) rz_head_features_kernel(const HeadsParams p, float* __restrict__ feat) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  __shared__ __align__(16) float s_w[6 * HEAD_C];
  for (int i = threadIdx.x; i < 6 * HEAD_C; i += blockDim.x) s_w[i] = p.w1x1[i];
  __syncthreads();
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)p.n_boards * p.P) return;
  const int b = (int)(idx / p.P), t = (int)(idx - (long long)b * p.P);
  const int y = t / p.S, x = t - y * p.S;
  float acc[6];
#pragma unroll
  for (int f = 0; f < 6; ++f) acc[f] = p.b1x1[f];
  if (x < p.W && y < p.H) conv1x1_position<true>(p.act, b, y * p.W + x, p.W, p.HW, p.S, p.P, s_w, acc);
  float* fo = feat + (size_t)b * (6 * p.P) + t;
#pragma unroll
  for (int f = 0; f < 6; ++f) fo[f * p.P] = fmaxf(acc[f], 0.0f);
}

size_t heads_smem(int HW, int AS) {
  return sizeof(float) * ((size_t)HEAD_NB * 6 * HW + (size_t)HEAD_NB * AS + HEAD_NB * 64 + 6 * HEAD_C);
}

}  // namespace

extern "C" int rz_net_conv3x3_f32(const float* in, const float* weight, const float* bias,
                                  const float* residual, float* out, int n_boards, int board_size,
                                  int c_in, int c_out, int relu, void* stream) {
  RZ_REQUIRE(in && weight && bias && out, "rz_net_conv3x3_f32: null argument");
  RZ_REQUIRE(board_size >= 1 && board_size <= RZ_MAX_BOARD, "rz_net_conv3x3_f32: board_size %d", board_size);
  RZ_REQUIRE(c_in >= 1 && c_out >= 1 && n_boards >= 0, "rz_net_conv3x3_f32: bad sizes");
  RZ_REQUIRE(in != out, "rz_net_conv3x3_f32: in-place convolution is not supported");
  const size_t smem = sizeof(float) * (size_t)board_size * board_size * c_in;
  RZ_REQUIRE(smem <= 200 * 1024, "rz_net_conv3x3_f32: input board needs %zu B of shared memory", smem);
  if (n_boards == 0) return 0;
  // the register-tiled kernel needs output channels in groups of 4 and 16-byte aligned tensors, and pays off when a
  // board keeps a 256-thread block busy (>= 512 thread tiles: 15x15 with 32+ channels, not 3x3) and there are enough
  // boards to fill the GPU; a handful of boards (the single-game API) stay on the scalar kernel, split over blocks
  const int HWs = board_size * board_size, ct4 = c_out >> 2;
  const bool vec_ok = (c_out & 3) == 0 && ((((uintptr_t)weight) | ((uintptr_t)bias) | ((uintptr_t)out) |
                                            ((uintptr_t)residual)) & 15) == 0;
  const int tp = !(vec_ok && n_boards >= 64) ? 0 : (ct4 * ((HWs + 3) / 4) >= 512 ? 4 : (ct4 * HWs >= 512 ? 1 : 0));
  const bool tiled = tp != 0;
  cudaError_t e = !tiled ? cudaFuncSetAttribute(rz_conv3x3_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                  : tp == 1 ? cudaFuncSetAttribute(rz_conv3x3_f32_tiled_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                            : cudaFuncSetAttribute(rz_conv3x3_f32_tiled_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { rz_set_error("rz_net_conv3x3_f32: smem attribute: %s", cudaGetErrorString(e)); return -2; }
  // few boards (the single-game API): split each board over several blocks so that the grid covers the 148 SMs
  int split = (2 * 148 + n_boards - 1) / n_boards;
  const int max_split = (board_size * board_size * c_out + 255) / 256;
  if (split > max_split) split = max_split;
  if (split > 64) split = 64;
  if (split < 1) split = 1;
  if (tiled) {
    const int tiles = (c_out >> 2) * ((board_size * board_size + tp - 1) / tp);
    if (split > (tiles + 255) / 256) split = (tiles + 255) / 256;
    if (tp == 1)
      rz_launch_pdl(rz_conv3x3_f32_tiled_kernel<1>, dim3((unsigned)n_boards, (unsigned)split), 256, smem, (cudaStream_t)stream, 
          in, weight, bias, residual, out, board_size, c_in, c_out, relu);
    else
      rz_launch_pdl(rz_conv3x3_f32_tiled_kernel<4>, dim3((unsigned)n_boards, (unsigned)split), 256, smem, (cudaStream_t)stream, 
          in, weight, bias, residual, out, board_size, c_in, c_out, relu);
  } else {
    rz_launch_pdl(rz_conv3x3_f32_kernel, dim3((unsigned)n_boards, (unsigned)split), 256, smem, (cudaStream_t)stream, 
        in, weight, bias, residual, out, board_size, c_in, c_out, relu);
  }
  RZ_LAUNCH_CHECK("rz_net_conv3x3_f32");
  return 0;
}

extern "C" int rz_net_heads(const rz_heads_desc* h, const float* act, float* logp, float* value, int n_boards,
                            void* stream) {
  RZ_REQUIRE(h && act && logp && value, "rz_net_heads: null argument");
  RZ_REQUIRE(h->w1x1 && h->b1x1 && h->wp && h->bp && h->wv1 && h->bv1 && h->wv2 && h->bv2,
             "rz_net_heads: null weight pointer");
  RZ_REQUIRE(h->board_size >= 1 && h->board_size <= RZ_MAX_BOARD, "rz_net_heads: board_size %d", h->board_size);
  const int W = h->width > 0 ? h->width : h->board_size;
  RZ_REQUIRE(W >= 1 && W <= RZ_MAX_BOARD, "rz_net_heads: width %d", W);
  const int HW = h->board_size * W;
  const int A = h->n_actions > 0 ? h->n_actions : HW;
  RZ_REQUIRE(h->action_stride >= A && (h->action_stride & 31) == 0, "rz_net_heads: action_stride %d", h->action_stride);
  if (n_boards <= 0) return 0;
  HeadsParams p;
  memset(&p, 0, sizeof(p));
  p.act = act; p.w1x1 = h->w1x1; p.b1x1 = h->b1x1; p.wp = h->wp; p.bp = h->bp; p.wv1 = h->wv1;
  p.bv1 = h->bv1; p.wv2 = h->wv2; p.bv2 = h->bv2; p.logp = logp; p.value = value;
  p.n_boards = n_boards; p.H = h->board_size; p.W = W; p.HW = HW; p.A = A; p.AS = h->action_stride;
  const size_t smem = heads_smem(HW, p.AS);
  cudaError_t e = cudaFuncSetAttribute(rz_heads_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { rz_set_error("rz_net_heads: smem attribute: %s", cudaGetErrorString(e)); return -2; }
  rz_launch_pdl(rz_heads_kernel, (n_boards + HEAD_NB - 1) / HEAD_NB, HEAD_THREADS, smem, (cudaStream_t)stream, p);
  RZ_LAUNCH_CHECK("rz_net_heads");
  return 0;
}

extern "C" int rz_net_head_features(const rz_heads_desc* h, const void* act, float* feat, int n_boards,
                                    void* stream) {
  RZ_REQUIRE(h && act && feat, "rz_net_head_features: null argument");
  RZ_REQUIRE(h->w1x1 && h->b1x1, "rz_net_head_features: null weight pointer");
  RZ_REQUIRE(h->board_size >= 1 && h->board_size <= RZ_MAX_BOARD, "rz_net_head_features: board_size %d", h->board_size);
  const int W = h->width > 0 ? h->width : h->board_size;
  RZ_REQUIRE(W >= 1 && W <= RZ_MAX_BOARD, "rz_net_head_features: width %d", W);
  const int S = rz_row_stride(h->board_size, W, h->row_stride);
  RZ_REQUIRE(S != 0, "rz_net_head_features: row_stride %d does not hold a %dx%d board", h->row_stride, h->board_size, W);
  if (n_boards <= 0) return 0;
  HeadsParams p;
  memset(&p, 0, sizeof(p));
  p.act = act; p.w1x1 = h->w1x1; p.b1x1 = h->b1x1;
  p.n_boards = n_boards; p.H = h->board_size; p.W = W; p.HW = h->board_size * W; p.S = S; p.P = S * S;
  const long long total = (long long)n_boards * p.P;
  rz_launch_pdl(rz_head_features_kernel, (unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream, p, feat);
  RZ_LAUNCH_CHECK("rz_net_head_features");
  return 0;
}
