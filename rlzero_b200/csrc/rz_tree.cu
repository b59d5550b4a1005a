// rlzero_b200 -- search-tree kernels: one warp owns one tree.
//
// Reference semantics (file:line under /root/reference):
//   select         rlzero/mcts/alphazero_mcts.py:48-54, rlzero/mcts/node.py:32-42,75-88
//   PUCT rule      rlzero/mcts/deepmind_mcts.py:149-151
//   expand         rlzero/mcts/node.py:44-73
//   terminal value rlzero/mcts/alphazero_mcts.py:60-68
//   backup         rlzero/mcts/node.py:119-144
//   root policy    rlzero/mcts/alphazero_mcts.py:86-94,144-148
//   re-root        rlzero/mcts/alphazero_mcts.py:96-103
//   trajectory     rlzero/games/gomoku/game.py:113-134
//
// Layout: an expanded node owns an "edge block" of AS slots indexed by action; a child's
// visit count / value sum live in its parent's block, so one descent step is one coalesced
// sweep over N (and W only when every child has been visited).  The reference runs one
// playout at a time; here every tree runs exactly one playout per wave, which keeps the
// per-tree order of updates -- and therefore every fp64 sum and every tie-break -- identical.
//
// Bit-exactness: scores are formed with the explicit round-to-nearest fp64 intrinsics
// (__ddiv_rn/__dsqrt_rn/__dmul_rn/__dadd_rn never contract into FMA), ln(Np) comes from a
// host-libm table (CPython's math.log), and ties go to the lowest action (Python max()).
#include <string.h>

#include "rz_board.cuh"
#include "rz_go.cuh"

#define RZ_TREE_WARPS 4
#define RZ_TREE_THREADS (RZ_TREE_WARPS * 32)
#define RZ_MAX_ITERS 12  // AS/32 <= 12  (A <= 362 -> AS <= 384)

__device__ __forceinline__ size_t rz_edge_base(const rz_tree_desc& t, int g, int node) {
  return ((size_t)g * t.max_nodes + node) * (size_t)t.game.action_stride;
}

// argmax over (score desc, slot asc) across the warp; n rides along.
__device__ __forceinline__ void rz_warp_argmax(double& s, int& slot, int& n) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double s2 = __shfl_xor_sync(RZ_FULL, s, o);
    const int slot2 = __shfl_xor_sync(RZ_FULL, slot, o);
    const int n2 = __shfl_xor_sync(RZ_FULL, n, o);
    const bool take = (slot2 >= 0) && (slot < 0 || s2 > s || (s2 == s && slot2 < slot));
    if (take) { s = s2; slot = slot2; n = n2; }
  }
}
// the same over (score desc, rank asc, slot asc): `rank` is the child's position in the parent's shuffled
// `children` list (deepmind_mcts.py:508), the order Python's max() breaks ties in
__device__ __forceinline__ void rz_warp_argmax_ranked(double& s, int& rank, int& slot, int& n) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double s2 = __shfl_xor_sync(RZ_FULL, s, o);
    const int r2 = __shfl_xor_sync(RZ_FULL, rank, o);
    const int slot2 = __shfl_xor_sync(RZ_FULL, slot, o);
    const int n2 = __shfl_xor_sync(RZ_FULL, n, o);
    const bool take = (slot2 >= 0) && (slot < 0 || s2 > s ||
                                       (s2 == s && (r2 < rank || (r2 == rank && slot2 < slot))));
    if (take) { s = s2; rank = r2; slot = slot2; n = n2; }
  }
}

// SearchNode.outcome codes (DeepMindMCTS flavour): 0 = None, else 0x100 | (o[0]+1) | (o[1]+1) << 2
__device__ __forceinline__ int rz_outcome_enc(int o0, int o1) { return 0x100 | (o0 + 1) | ((o1 + 1) << 2); }
__device__ __forceinline__ int rz_outcome_of(int code, int player) { return ((code >> (2 * player)) & 3) - 1; }

// ---------------------------------------------------------------------------
// K1: select.  One playout descent per tree + leaf terminal test.
// ---------------------------------------------------------------------------
// one descent of tree g; its path / leaf go to wave slot L (= g in the parity mode, g*K + k in leaf-parallel mode)
template <class GM, bool DM>
__device__ __forceinline__ void rz_select_one(const rz_tree_desc& t, const int g, const int L, const rz_geom& q,
                                              int32_t* rmeta) {
  const int lane = rz_lane();
  const int AS = t.game.action_stride;
  const int iters = AS >> 5;
  typename GM::board b;
  GM::load_root(b, t, g);
  const int root_player = b.player;

  int fault = 0;
  int depth = 0;
  int node = 0;
  int Np = t.root_N[g];
  bool descend = t.n_nodes[g] > 0;
  int32_t* pnode = t.path_node + (size_t)L * t.max_depth;
  int32_t* pact = t.path_action + (size_t)L * t.max_depth;

  while (descend) {
    if (depth >= t.max_depth) { fault |= RZ_FAULT_DEPTH_OVERFLOW; break; }
    const size_t base = rz_edge_base(t, g, node);
    const int32_t* eN = t.edge_N + base;
    // pass 1: visit counts (coalesced, all loads in flight at once)
    int nv[RZ_MAX_ITERS];
#pragma unroll
    for (int i = 0; i < RZ_MAX_ITERS; ++i) nv[i] = (i < iters) ? eN[lane + 32 * i] : -1;

    double best_s = 0.0;
    int best_slot = -1, best_n = 0, best_r = 0;
    // DeepMindMCTS with the child shuffle: ties go to the child that comes first in the shuffled list
    const bool ranked = DM && t.edge_R != nullptr;
    int rk[RZ_MAX_ITERS];
    if (ranked) {
      const int32_t* eR = t.edge_R + base;
#pragma unroll
      for (int i = 0; i < RZ_MAX_ITERS; ++i) rk[i] = (i < iters && nv[i] >= 0) ? eR[lane + 32 * i] : 0x7fffffff;
    }
    // DeepMindMCTS: a child with a known outcome scores outcome[child.player] (deepmind_mcts.py:123-124,
    // 146-147); the children of a node at this depth were all moved by the same player
    int oc[RZ_MAX_ITERS];
    const int mover = root_player ^ (depth & 1);
    if (DM) {
      const int32_t* eO = t.edge_O + base;
#pragma unroll
      for (int i = 0; i < RZ_MAX_ITERS; ++i) oc[i] = (i < iters && nv[i] > 0) ? eO[lane + 32 * i] : 0;
    }
    if (t.rule == RZ_RULE_UCT) {
      // node.py:76-80: +inf when the parent or the child is unvisited -> first such child wins
      int first_unvisited = -1;
#pragma unroll
      for (int i = RZ_MAX_ITERS - 1; i >= 0; --i)
        if (i < iters && (nv[i] == 0 || (nv[i] > 0 && Np == 0))) first_unvisited = lane + 32 * i;
      // lowest slot over the warp
      int cand = first_unvisited < 0 ? 0x7fffffff : first_unvisited;
      if (ranked) {
        // every unvisited child scores +inf: the first of them in list order wins
        long long key = 0x7fffffffffffffffll;
#pragma unroll
        for (int i = 0; i < RZ_MAX_ITERS; ++i)
          if (i < iters && (nv[i] == 0 || (nv[i] > 0 && Np == 0))) {
            const long long k2 = ((long long)rk[i] << 32) | (unsigned)(lane + 32 * i);
            key = k2 < key ? k2 : key;
          }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const long long k2 = __shfl_xor_sync(RZ_FULL, key, o);
          key = k2 < key ? k2 : key;
        }
        cand = key == 0x7fffffffffffffffll ? 0x7fffffff : (int)(key & 0xffffffffll);
      } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(RZ_FULL, cand, o));
      }
      if (cand != 0x7fffffff) {
        best_slot = cand;
        best_n = eN[cand];
      } else {
        // every child visited: W/n + c*sqrt(ln(Np)/n)   (node.py:82-88)
        const double* eW = t.edge_W + base;
        double wv[RZ_MAX_ITERS];
#pragma unroll
        for (int i = 0; i < RZ_MAX_ITERS; ++i)
          wv[i] = (i < iters && nv[i] > 0) ? eW[lane + 32 * i] : 0.0;
        int NpC = Np;
        if (NpC >= t.ln_table_len) { fault |= RZ_FAULT_LN_TABLE; NpC = t.ln_table_len - 1; }
        const double lnNp = t.ln_table[NpC];
#pragma unroll
        for (int i = 0; i < RZ_MAX_ITERS; ++i) {
          if (i < iters && nv[i] > 0) {
            const double n = (double)nv[i];
            const double q = __ddiv_rn(wv[i], n);
            const double u = __dsqrt_rn(__ddiv_rn(lnNp, n));
            double s = __dadd_rn(q, __dmul_rn(t.c_puct, u));
            if (DM && oc[i]) s = (double)rz_outcome_of(oc[i], mover);
            if (best_slot < 0 || s > best_s || (ranked && s == best_s && rk[i] < best_r)) {
              best_s = s; best_slot = lane + 32 * i; best_n = nv[i]; best_r = ranked ? rk[i] : 0;
            }
          }
        }
        if (ranked) rz_warp_argmax_ranked(best_s, best_r, best_slot, best_n);
        else rz_warp_argmax(best_s, best_slot, best_n);
      }
    } else {
      // deepmind_mcts.py:149-151: (n and W/n) + ((c*P)*sqrt(Np))/(n+1)
      const double* eW = t.edge_W + base;
      const float* eP = t.edge_P + base;
      const double* eP64 = t.edge_P64 ? t.edge_P64 + base : nullptr;   // float64 priors (noise mixed in float64)
      const double sq = __dsqrt_rn((double)Np);
#pragma unroll
      for (int i = 0; i < RZ_MAX_ITERS; ++i) {
        if (i < iters && nv[i] >= 0) {
          const int slot = lane + 32 * i;
          const double q = nv[i] > 0 ? __ddiv_rn(eW[slot], (double)nv[i]) : 0.0;
          const double pr = eP64 ? eP64[slot] : (double)eP[slot];
          const double u = __ddiv_rn(__dmul_rn(__dmul_rn(t.c_puct, pr), sq), (double)(nv[i] + 1));
          double s = __dadd_rn(q, u);
          if (DM && oc[i]) s = (double)rz_outcome_of(oc[i], mover);
          if (best_slot < 0 || s > best_s || (ranked && s == best_s && rk[i] < best_r)) {
            best_s = s; best_slot = slot; best_n = nv[i]; best_r = ranked ? rk[i] : 0;
          }
        }
      }
      if (ranked) rz_warp_argmax_ranked(best_s, best_r, best_slot, best_n);
      else rz_warp_argmax(best_s, best_slot, best_n);
    }
    if (best_slot < 0) { fault |= RZ_FAULT_NO_CHILDREN; break; }  // node.py:38-39

    if (lane == 0) { pnode[depth] = node; pact[depth] = best_slot; }
    depth += 1;
    GM::play(b, best_slot, q);       // game_env.step(action), alphazero_mcts.py:54
    if (best_n == 0) break;          // never visited -> unexpanded leaf
    const int child = t.edge_child[base + best_slot];
    if (child < 0) break;            // terminal (or overflowed) leaf, re-evaluated every visit
    node = child;
    Np = best_n;
  }

  // leaf: game_end_winner() (alphazero_mcts.py:60)
  int winner;
  const int status = GM::status(b, q, winner);
  GM::store_leaf(b, t, L);
  if (lane == 0) {
    int32_t* lm = t.leaf_meta + (size_t)L * RZ_META_STRIDE;
    GM::store_meta(b, lm);
    lm[RZ_META_STATUS] = status;
    lm[RZ_META_WINNER] = winner;
    lm[RZ_META_PLY] = depth;
    lm[RZ_META_FAULT] = fault;
    lm[RZ_META_EPISODE] = rmeta[RZ_META_EPISODE];
    t.depth[L] = depth;
    if (fault) rmeta[RZ_META_FAULT] |= fault;
  }
}

template <class GM, bool DM>
__global__ void __launch_bounds__(RZ_TREE_THREADS) rz_select_kernel(rz_tree_desc t) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  const int g = blockIdx.x * RZ_TREE_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  const int lane = rz_lane();
  const rz_geom q = rz_geom_of(t.game);
  const int K = t.leaves_per_tree > 1 ? t.leaves_per_tree : 1;
  int32_t* rmeta = t.root_meta + (size_t)g * RZ_META_STRIDE;
  // a finished game, or (DeepMindMCTS) a proven root: `if root.outcome is not None: break` (:643-644)
  if (rmeta[RZ_META_STATUS] != RZ_ACTIVE || (DM && t.root_O[g] != 0)) {
    for (int k = lane; k < K; k += 32) t.depth[(size_t)g * K + k] = -1;
    return;
  }
  if (K == 1) {                      // the parity mode: the reference's strictly sequential playouts
    rz_select_one<GM, DM>(t, g, g, q, rmeta);
    return;
  }
  // leaf-parallel wave: up to K descents, each followed by its virtual loss (see rz_tree_desc.leaves_per_tree)
  int budget = K;
  if (t.target_N) budget = min(budget, t.target_N[g] - t.root_N[g]);
  if (t.n_nodes[g] == 0) budget = min(budget, 1);      // the first playout only expands the root
  for (int k = 0; k < K; ++k) {
    const int L = g * K + k;
    if (k >= budget) {
      if (lane == 0) t.depth[L] = -1;
      continue;
    }
    rz_select_one<GM, DM>(t, g, L, q, rmeta);
    __syncwarp();
    const int depth = t.depth[L];
    const int32_t* pnode = t.path_node + (size_t)L * t.max_depth;
    const int32_t* pact = t.path_action + (size_t)L * t.max_depth;
    double* saved = t.vl_saved_W + (size_t)L * t.max_depth;
    for (int i = lane; i < depth; i += 32) {
      const size_t e = rz_edge_base(t, g, pnode[i]) + pact[i];
      const int n = t.edge_N[e];
      const double w = t.edge_W[e];
      saved[i] = w;
      t.edge_W[e] = n > 0 ? __dadd_rn(w, -t.virtual_loss) : -t.virtual_loss;
      t.edge_N[e] = n + 1;
      if (n == 0) t.edge_child[e] = RZ_CHILD_PENDING;   // visited only virtually: a later descent stops here
    }
    if (lane == 0) t.root_N[g] += 1;
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Dirichlet(alpha) noise: one Gamma(alpha,1) draw per legal slot, normalised over the node (node.py:63-69).
// alpha < 1 (the reference's 0.3): Ahrens-Dieter GS rejection sampler -- two uniforms and two exp/log-class
// evaluations per attempt, acceptance e*Gamma(alpha+1)/(e+alpha) = 0.81 at alpha = 0.3, two attempts per Philox
// call.  (The expansion kernel spent most of its instructions here: 225 draws per tree and wave with the
// Marsaglia-Tsang + boost sampler kept below for alpha >= 1 -- a normal, three logs and a pow per attempt.)
// ---------------------------------------------------------------------------
__device__ float rz_gamma_draw(float alpha, unsigned long long seed, uint32_t c0, uint32_t c1,
                               uint32_t c2) {
  if (alpha < 1.0f) {
    const float inv_a = 1.0f / alpha, b = 1.0f + alpha * 0.36787944117f;
    for (uint32_t it = 0; it < 32; ++it) {
      uint32_t r[4];
      rz_philox4(c0, c1, c2, it, seed, r);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float p = b * rz_u01_24(r[2 * h]), u2 = rz_u01_24(r[2 * h + 1]);
        float x, bound;
        if (p <= 1.0f) {
          x = __powf(p, inv_a);                       // density ~ x^(alpha-1) on (0,1], accept with e^-x
          bound = __expf(-x);
        } else {
          x = -__logf((b - p) * inv_a);               // density ~ e^-x on (1,inf), accept with x^(alpha-1)
          bound = __powf(x, alpha - 1.0f);
        }
        if (u2 <= bound) return x;
      }
    }
    return alpha;  // unreachable in practice (0.19^64)
  }
  const float d = alpha + 1.0f - 1.0f / 3.0f;
  const float c = rsqrtf(9.0f * d);
  for (uint32_t it = 0; it < 64; ++it) {
    uint32_t r[4];
    rz_philox4(c0, c1, c2, it, seed, r);
    // Box-Muller normal from r[0], r[1]
    const float u1 = rz_u01_24(r[0]), u2 = rz_u01_24(r[1]);
    const float x = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
    float v = 1.0f + c * x;
    if (v <= 0.0f) continue;
    v = v * v * v;
    const float u = rz_u01_24(r[2]);
    if (logf(u) < 0.5f * x * x + d - d * v + d * logf(v)) {
      const float boost = powf(rz_u01_24(r[3]), 1.0f / alpha);
      return d * v * boost;
    }
  }
  return alpha;  // unreachable in practice
}

// ---------------------------------------------------------------------------
// K5+K6: expand the leaf (unless terminal) and back the value up the path.
// ---------------------------------------------------------------------------
// leaf slot L of tree g (L = g in the parity mode).  `dedup`: leaf-parallel mode, where a leaf may have been
// expanded by an earlier playout of the same wave.
template <class GM, bool DM>
__device__ __forceinline__ void
rz_expand_backup_one(const rz_tree_desc& t, const int g, const int L, const bool dedup, const rz_geom& q,
                     const float* prior, int prior_is_log, const float* value, const double* value64,
                     float noise_eps, float noise_alpha, unsigned long long seed, long long global_offset,
                     const double* noise64, const double* prior64) {
  const int depth = t.depth[L];
  if (depth < 0) return;
  const int lane = rz_lane();
  const int AS = t.game.action_stride;
  const int32_t* lm = t.leaf_meta + (size_t)L * RZ_META_STRIDE;
  const int32_t* rm = t.root_meta + (size_t)g * RZ_META_STRIDE;
  const int status = lm[RZ_META_STATUS];
  int32_t* pnode = t.path_node + (size_t)L * t.max_depth;
  int32_t* pact = t.path_action + (size_t)L * t.max_depth;

  // alphazero_mcts.py:59-68: network value unless the game is over at the leaf
  double v;
  int child_mark = 0;  // what to store in the parent's child[] slot
  bool have_mark = false;
  if (status == RZ_ENDED_WIN) {
    v = (lm[RZ_META_WINNER] == lm[RZ_META_PLAYER]) ? 1.0 : -1.0;
    child_mark = RZ_CHILD_TERMINAL; have_mark = true;
  } else if (status == RZ_ENDED_TIE) {
    v = 0.0;
    child_mark = RZ_CHILD_TERMINAL; have_mark = true;
  } else {
    v = value64 ? value64[L] : (double)value[L];
    const int nn = t.n_nodes[g];
    // leaf-parallel mode: an earlier playout of this wave reached the same leaf and expanded it already
    const bool expanded_already =
        dedup && (depth > 0 ? t.edge_child[rz_edge_base(t, g, pnode[depth - 1]) + pact[depth - 1]] >= 0 : nn > 0);
    if (expanded_already) {
      // back the (identical) evaluation up once more, nothing to create
    } else if (nn < t.max_nodes) {
      // node.py:71-73: one child per legal move, in ascending action order
      const uint32_t lctx = GM::legal_ctx(t, L, q);
      const size_t nb = rz_edge_base(t, g, nn);
      const float* pr = prior ? prior + (size_t)L * AS : nullptr;
      float noise_sum = 0.0f;
      float nz[RZ_MAX_ITERS];
      // host-supplied randomness (rz_tree_expand_backup_ex): no device draw
      const double* hn = noise64 ? noise64 + (size_t)L * AS : nullptr;
      const double* hp = prior64 ? prior64 + (size_t)L * AS : nullptr;
      // the UCB1 rule never reads a prior: with no prior pool there is nothing the noise could change
      const bool noisy = noise_eps > 0.0f && !(DM && t.noise_root_only && depth > 0) && !hp && t.store_priors;
      const bool draw = noisy && !hn;
      // noise stream of this node: Philox counter (global game, episode | slot << 20, ply << 16 | node, attempt)
      const uint32_t c1 = (uint32_t)rm[RZ_META_EPISODE] & 0xfffffu;
      const uint32_t c2 = ((uint32_t)rm[RZ_META_PLY] << 16) | (uint32_t)nn;
#pragma unroll
      for (int i = 0; i < RZ_MAX_ITERS; ++i) {
        if (i >= (AS >> 5)) break;
        const int s = lane + 32 * i;
        const bool legal = GM::slot_legal(lctx, s, q);
        t.edge_N[nb + s] = legal ? 0 : -1;
        if (DM) t.edge_O[nb + s] = 0;
        if (DM && t.edge_R) {
          // children order: a random key per child (a uniformly random order, ties broken by the action), or the
          // slot itself when the host supplies numpy's permutation afterwards (rz_tree_desc.edge_R)
          int r = s;
          if (t.shuffle_mode == 1) {
            uint32_t rr[4];
            rz_philox4((uint32_t)(global_offset + g), c1 | ((uint32_t)s << 20), c2, 0xffffu,
                       seed ^ 0x517cc1b727220a95ull, rr);
            r = (int)(rr[0] >> 1);
          }
          t.edge_R[nb + s] = legal ? r : 0x7fffffff;
        }
        nz[i] = 0.0f;
        if (draw && legal) {
          nz[i] = rz_gamma_draw(noise_alpha, seed, (uint32_t)(global_offset + g), c1 | ((uint32_t)s << 20), c2);
          noise_sum += nz[i];
        }
        if (hp) {
          const double p = legal ? hp[s] : 0.0;
          if (t.store_priors) t.edge_P[nb + s] = (float)p;
          if (t.edge_P64) t.edge_P64[nb + s] = p;
        } else if (t.store_priors && !noisy) {
          float p = legal ? pr[s] : 0.0f;
          if (legal && prior_is_log) p = expf(p);
          t.edge_P[nb + s] = p;
          if (t.edge_P64) t.edge_P64[nb + s] = (double)p;
        }
      }
      if (noisy) {
        float inv = 0.0f;
        if (draw) {
          noise_sum = rz_warp_sum_f32(noise_sum);
          inv = noise_sum > 0.0f ? 1.0f / noise_sum : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < RZ_MAX_ITERS; ++i) {
          if (i >= (AS >> 5)) break;
          const int s = lane + 32 * i;
          const bool legal = t.edge_N[nb + s] == 0;
          float p = legal ? pr[s] : 0.0f;
          if (legal && prior_is_log) p = expf(p);
          if (hn) {
            // numpy: float32 * python float stays float32, float32 + float64 is float64 (node.py:68)
            const double mixed = legal ? __dadd_rn((double)__fmul_rn(1.0f - noise_eps, p),
                                                   __dmul_rn((double)noise_eps, hn[s])) : 0.0;
            t.edge_P[nb + s] = (float)mixed;
            if (t.edge_P64) t.edge_P64[nb + s] = mixed;
          } else {
            const float mixed = legal ? (1.0f - noise_eps) * p + noise_eps * nz[i] * inv : 0.0f;
            t.edge_P[nb + s] = mixed;
            if (t.edge_P64) t.edge_P64[nb + s] = (double)mixed;
          }
        }
      }
      if (lane == 0) {
        t.node_parent[(size_t)g * t.max_nodes + nn] = depth > 0 ? pnode[depth - 1] : -1;
        t.node_paction[(size_t)g * t.max_nodes + nn] = depth > 0 ? pact[depth - 1] : -1;
        t.n_nodes[g] = nn + 1;
      }
      child_mark = nn; have_mark = true;
    } else {
      child_mark = RZ_CHILD_OVERFLOW; have_mark = true;
      if (lane == 0) t.root_meta[(size_t)g * RZ_META_STRIDE + RZ_META_FAULT] |= RZ_FAULT_POOL_OVERFLOW;
    }
  }
  if (have_mark && depth > 0 && lane == 0) {
    t.edge_child[rz_edge_base(t, g, pnode[depth - 1]) + pact[depth - 1]] = child_mark;
  }

  if (DM) {
    // deepmind_mcts.py:596-644.  returns: env.returns() at a terminal leaf, else the evaluation
    // ([v,-v] in the order (player to move at the leaf, the other), or the evaluator's own vector);
    // every node on the path adds returns[node.player], node.player = who moved into it
    const int rp = rm[RZ_META_PLAYER];
    double ret[2];
    int code = 0;
    if (status != RZ_ACTIVE) {
      int r0, r1;
      rz_game_returns(t.game.game_type, t.returns_mode, status, lm[RZ_META_WINNER], r0, r1);
      ret[0] = (double)r0; ret[1] = (double)r1;
      code = rz_outcome_enc(r0, r1);
    } else if (value64) {                  // here: the evaluator's returns vector [G][2]
      ret[0] = value64[2 * L]; ret[1] = value64[2 * L + 1];
    } else {
      const int pl = lm[RZ_META_PLAYER] & 1;
      ret[pl] = v; ret[pl ^ 1] = -v;
    }
    for (int k = lane; k < depth; k += 32) {
      const size_t e = rz_edge_base(t, g, pnode[k]) + pact[k];
      const double x = ret[(rp ^ (k & 1)) & 1];
      const int n = t.edge_N[e];
      t.edge_W[e] = n > 0 ? __dadd_rn(t.edge_W[e], x) : __dadd_rn(0.0, x);
      t.edge_N[e] = n + 1;
    }
    if (lane == 0) {
      t.root_W[g] = __dadd_rn(t.root_W[g], ret[rp & 1]);
      t.root_N[g] += 1;
    }
    if (code) {
      // visit_path[-1].outcome = returns (:599), then MCTS-Solver up the path (:617-642)
      if (lane == 0) {
        if (depth == 0) t.root_O[g] = code;
        else t.edge_O[rz_edge_base(t, g, pnode[depth - 1]) + pact[depth - 1]] = code;
      }
      __syncwarp();
      bool solved = t.solve != 0;
      for (int d = depth - 1; solved && d >= 0; --d) {
        const size_t nb = rz_edge_base(t, g, pnode[d]);
        const int mover = (rp ^ (d & 1)) & 1;          // node.children[0].player
        int best_o = -2, best_slot = 0x7fffffff, best_code = 0;
        bool all_solved = true;
        for (int s = lane; s < AS; s += 32) {
          if (t.edge_N[nb + s] < 0) continue;          // not a child
          const int c = t.edge_O[nb + s];
          if (c == 0) { all_solved = false; continue; }
          const int o = rz_outcome_of(c, mover);
          if (o > best_o) { best_o = o; best_slot = s; best_code = c; }   // first maximum per lane (s ascends)
        }
        all_solved = __all_sync(RZ_FULL, all_solved);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          const int o2 = __shfl_xor_sync(RZ_FULL, best_o, off);
          const int s2 = __shfl_xor_sync(RZ_FULL, best_slot, off);
          const int c2 = __shfl_xor_sync(RZ_FULL, best_code, off);
          if (o2 > best_o || (o2 == best_o && s2 < best_slot)) { best_o = o2; best_slot = s2; best_code = c2; }
        }
        if (best_o > -2 && (all_solved || best_o == 1)) {              // max_utility() == 1
          if (lane == 0) {
            if (d == 0) t.root_O[g] = best_code;
            else t.edge_O[rz_edge_base(t, g, pnode[d - 1]) + pact[d - 1]] = best_code;
          }
          __syncwarp();
        } else {
          solved = false;
        }
      }
    }
  } else {
    // node.py:135-144 with update_recursive(-leaf_value): the leaf gets -v, its parent +v, ...
    // edge k (0-based from the root) holds the node at depth k+1 and gets (-1)^(depth-k) * v.
    for (int k = lane; k < depth; k += 32) {
      const size_t e = rz_edge_base(t, g, pnode[k]) + pact[k];
      const double x = ((depth - k) & 1) ? -v : v;
      const int n = t.edge_N[e];
      t.edge_W[e] = n > 0 ? __dadd_rn(t.edge_W[e], x) : __dadd_rn(0.0, x);
      t.edge_N[e] = n + 1;
    }
    if (lane == 0) {
      const double x = (depth & 1) ? v : -v;  // root at depth 0: (-1)^(depth+1) * v
      t.root_W[g] = __dadd_rn(t.root_W[g], x);
      t.root_N[g] += 1;
    }
  }
}

template <class GM, bool DM>
// 6 blocks (24 warps) per SM: 80 registers instead of 116; the kernel is latency-bound (16 warps/SM kept the issue
// slots 42 % busy), a few bytes of spill are the price
__global__ void __launch_bounds__(RZ_TREE_THREADS, 6)
rz_expand_backup_kernel(rz_tree_desc t, const float* __restrict__ prior, int prior_is_log,
                        const float* __restrict__ value, const double* __restrict__ value64,
                        float noise_eps, float noise_alpha,
                        unsigned long long seed, long long global_offset,
                        const double* __restrict__ noise64, const double* __restrict__ prior64) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  const int g = blockIdx.x * RZ_TREE_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  const rz_geom q = rz_geom_of(t.game);
  const int K = t.leaves_per_tree > 1 ? t.leaves_per_tree : 1;
  if (t.seed_dev) seed += *t.seed_dev;       // a captured graph draws fresh noise on every replay
  if (K == 1) {
    rz_expand_backup_one<GM, DM>(t, g, g, false, q, prior, prior_is_log, value, value64, noise_eps, noise_alpha, seed,
                                 global_offset, noise64, prior64);
    return;
  }
  // leaf-parallel wave: take the virtual losses off again -- the saved value sums in reverse order of application,
  // so every edge returns to its exact pre-wave bits -- then expand and back up the K leaves in order
  const int lane = rz_lane();
  for (int k = K - 1; k >= 0; --k) {
    const int L = g * K + k;
    const int depth = t.depth[L];
    if (depth < 0) continue;
    const int32_t* pnode = t.path_node + (size_t)L * t.max_depth;
    const int32_t* pact = t.path_action + (size_t)L * t.max_depth;
    const double* saved = t.vl_saved_W + (size_t)L * t.max_depth;
    for (int i = lane; i < depth; i += 32) {
      const size_t e = rz_edge_base(t, g, pnode[i]) + pact[i];
      t.edge_W[e] = saved[i];
      t.edge_N[e] -= 1;
    }
    if (lane == 0) t.root_N[g] -= 1;
    __syncwarp();
  }
  for (int k = 0; k < K; ++k) {
    rz_expand_backup_one<GM, DM>(t, g, g * K + k, true, q, prior, prior_is_log, value, value64, noise_eps, noise_alpha,
                                 seed, global_offset, noise64, prior64);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Expand + backup of wave w followed, in the same launch, by the selection of wave w + 1 (one leaf per tree and wave
// only).  The two halves belong to the same warp and the same tree, so nothing but a warp barrier lies between them:
// one launch and one kernel boundary less per wave, and the root's edge blocks the backup just touched are still in
// cache for the descent.  It matters where a wave is a handful of short kernels (a single game: ~5 us of ~50).
// ---------------------------------------------------------------------------
template <class GM, bool DM>
__global__ void __launch_bounds__(RZ_TREE_THREADS)
rz_expand_backup_select_kernel(rz_tree_desc t, const float* __restrict__ prior, int prior_is_log,
                               const float* __restrict__ value, const double* __restrict__ value64,
                               float noise_eps, float noise_alpha, unsigned long long seed, long long global_offset) {
  rz::grid_dep_wait();     // programmatic dependent launch: see rz_common.cuh
  rz::grid_dep_launch();
  const int g = blockIdx.x * RZ_TREE_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  const rz_geom q = rz_geom_of(t.game);
  if (t.seed_dev) seed += *t.seed_dev;
  rz_expand_backup_one<GM, DM>(t, g, g, false, q, prior, prior_is_log, value, value64, noise_eps, noise_alpha, seed,
                               global_offset, nullptr, nullptr);
  __syncwarp();            // the lanes read each other's updates of the path below
  int32_t* rmeta = t.root_meta + (size_t)g * RZ_META_STRIDE;
  if (rmeta[RZ_META_STATUS] != RZ_ACTIVE || (DM && t.root_O[g] != 0)) {
    if (rz_lane() == 0) t.depth[g] = -1;
    return;
  }
  rz_select_one<GM, DM>(t, g, g, q, rmeta);
}

// ---------------------------------------------------------------------------
// K7: root policy  pi = softmax(log(N + 1e-10) / T) over the root's children and move sampling
// (alphazero_mcts.py:86-94, 144-148).  Sampling mirrors numpy.random.choice: first index
// whose normalised cumulative probability exceeds u.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(RZ_TREE_THREADS)
rz_root_policy_kernel(rz_tree_desc t, double temperature, int32_t* __restrict__ visits,
                      float* __restrict__ pi, int32_t* __restrict__ move,
                      const double* __restrict__ u01, unsigned long long seed,
                      long long global_offset) {
  const int g = blockIdx.x * RZ_TREE_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  const int lane = rz_lane();
  const int AS = t.game.action_stride;
  const int iters = AS >> 5;
  int32_t* rmeta = t.root_meta + (size_t)g * RZ_META_STRIDE;
  const bool active = rmeta[RZ_META_STATUS] == RZ_ACTIVE;
  const bool expanded = t.n_nodes[g] > 0;
  const size_t base = rz_edge_base(t, g, 0);
  int nv[RZ_MAX_ITERS];
  double x[RZ_MAX_ITERS];
  double mx = -1.0e300;
#pragma unroll
  for (int i = 0; i < RZ_MAX_ITERS; ++i) {
    nv[i] = (i < iters && active && expanded) ? t.edge_N[base + lane + 32 * i] : -1;
    x[i] = 0.0;
    if (nv[i] >= 0) {
      x[i] = (1.0 / temperature) * log((double)nv[i] + 1e-10);
      mx = fmax(mx, x[i]);
    }
  }
  mx = rz_warp_max_f64(mx);
  double sum = 0.0;
#pragma unroll
  for (int i = 0; i < RZ_MAX_ITERS; ++i) {
    x[i] = nv[i] >= 0 ? exp(x[i] - mx) : 0.0;
    sum += x[i];
  }
  sum = rz_warp_sum_f64(sum);
  const bool any = sum > 0.0;
  if (active && !any && lane == 0) rmeta[RZ_META_FAULT] |= RZ_FAULT_NO_CHILDREN;
#pragma unroll
  for (int i = 0; i < RZ_MAX_ITERS; ++i) {
    if (i < iters) {
      const size_t o = (size_t)g * AS + lane + 32 * i;
      x[i] = any ? x[i] / sum : 0.0;
      if (visits) visits[o] = nv[i] > 0 ? nv[i] : 0;
      if (pi) pi[o] = (float)x[i];
    }
  }
  if (move) {
    double u;
    if (u01) {
      u = u01[g];
    } else {
      uint32_t r[4];
      rz_philox4((uint32_t)(global_offset + g), (uint32_t)rmeta[RZ_META_EPISODE],
                 (uint32_t)rmeta[RZ_META_STONES], 0x5eedu, seed, r);
      u = rz_u01_53(r[0], r[1]);
    }
    // cumulative sum in action order: slot = lane + 32*i, so scan chunk by chunk
    int chosen = -1, last_legal = -1;
    double carry = 0.0;
    for (int i = 0; i < iters; ++i) {
      double xi = 0.0; int ni = -1;
#pragma unroll
      for (int j = 0; j < RZ_MAX_ITERS; ++j) if (j == i) { xi = x[j]; ni = nv[j]; }
      const double inc = rz_warp_scan_f64(xi) + carry;
      const unsigned hit = __ballot_sync(RZ_FULL, ni >= 0 && inc > u);
      const unsigned leg = __ballot_sync(RZ_FULL, ni >= 0);
      if (leg) last_legal = 32 * i + (31 - __clz(leg));
      if (hit && chosen < 0) chosen = 32 * i + (__ffs(hit) - 1);
      carry = __shfl_sync(RZ_FULL, inc, 31);
    }
    if (chosen < 0) chosen = last_legal;  // u beyond the rounded total
    if (lane == 0) move[g] = (active && any) ? chosen : -1;
  }
}

// ---------------------------------------------------------------------------
// K8 (+K9): play the move on the root position, record the trajectory ply, re-root.
// ---------------------------------------------------------------------------
extern __shared__ uint32_t rz_adv_smem[];

__device__ void rz_tree_fresh(const rz_tree_desc& t, int g, int n, double w) {
  t.n_nodes[g] = 0;
  t.root_N[g] = n;
  t.root_W[g] = w;
  if (t.root_O) t.root_O[g] = 0;
}

__device__ __forceinline__ int rz_newidx(const uint32_t* bits, const uint32_t* wprefix, int i) {
  return (int)wprefix[i >> 5] + __popc(bits[i >> 5] & ((1u << (i & 31)) - 1u));
}

// In-place compaction of the subtree rooted at old node c to indices 0..m-1, ascending
// old index (parents always precede children, so dst <= src and nothing unread is clobbered).
__device__ int rz_tree_compact(const rz_tree_desc& t, int g, int c, uint32_t* bits,
                               uint32_t* wprefix, int max_carry) {
  const int lane = rz_lane();
  const int nn = t.n_nodes[g];
  const int nwords = (nn + 31) >> 5;
  const int AS = t.game.action_stride;
  int32_t* parent = t.node_parent + (size_t)g * t.max_nodes;
  int32_t* paction = t.node_paction + (size_t)g * t.max_nodes;
  for (int w = lane; w < nwords; w += 32) bits[w] = 0u;
  __syncwarp();
  // 1. membership sweep
  for (int i0 = (c >> 5) << 5; i0 < nn; i0 += 32) {
    const int i = i0 + lane;
    const int p = i < nn ? parent[i] : -1;
    bool in = (i == c);
    if (i < nn && i > c && p >= 0 && p < i0) in = (bits[p >> 5] >> (p & 31)) & 1u;
    const bool local = (i < nn && i > c && p >= i0);
    for (int it = 0; it < 32; ++it) {
      const bool pin = __shfl_sync(RZ_FULL, in, local ? (p - i0) : 0);
      const bool nin = in || (local && pin);
      const unsigned changed = __ballot_sync(RZ_FULL, nin != in);
      in = nin;
      if (!changed) break;
    }
    const unsigned word = __ballot_sync(RZ_FULL, in);
    if (lane == 0) bits[i0 >> 5] = word;
    __syncwarp();
  }
  // 2. exclusive prefix of popcounts per word
  int total = 0;
  for (int w0 = 0; w0 < nwords; w0 += 32) {
    const int w = w0 + lane;
    const int cnt = w < nwords ? __popc(bits[w]) : 0;
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int tt = __shfl_up_sync(RZ_FULL, inc, o);
      if (lane >= o) inc += tt;
    }
    if (w < nwords) wprefix[w] = total + inc - cnt;
    total += __shfl_sync(RZ_FULL, inc, 31);
  }
  __syncwarp();
  if (total > max_carry) return -1;
  // 3. move blocks
  for (int w = c >> 5; w < nwords; ++w) {
    uint32_t word = bits[w];
    while (word) {
      const int bit = __ffs(word) - 1;
      word &= word - 1;
      const int src = (w << 5) + bit;
      const int dst = rz_newidx(bits, wprefix, src);
      const size_t sb = rz_edge_base(t, g, src), db = rz_edge_base(t, g, dst);
      for (int s = lane; s < AS; s += 32) {
        const int n = t.edge_N[sb + s];
        const double wv = t.edge_W[sb + s];
        int ch = t.edge_child[sb + s];
        if (n >= 1 && ch >= 0) ch = rz_newidx(bits, wprefix, ch);
        t.edge_N[db + s] = n;
        t.edge_W[db + s] = wv;
        t.edge_child[db + s] = ch;
        if (t.store_priors) t.edge_P[db + s] = t.edge_P[sb + s];
        if (t.edge_P64) t.edge_P64[db + s] = t.edge_P64[sb + s];
        if (t.edge_O) t.edge_O[db + s] = t.edge_O[sb + s];
        if (t.edge_R) t.edge_R[db + s] = t.edge_R[sb + s];
      }
      if (lane == 0) {
        const int p = parent[src];
        const int pa = paction[src];
        parent[dst] = (src == c) ? -1 : rz_newidx(bits, wprefix, p);
        paction[dst] = (src == c) ? -1 : pa;
      }
      __syncwarp();
    }
  }
  return total;
}

template <class GM>
__global__ void __launch_bounds__(RZ_TREE_THREADS)
rz_advance_kernel(rz_tree_desc t, const int32_t* __restrict__ moves, int keep_subtree,
                  int max_carry, rz_traj_desc traj, int have_traj, const float* __restrict__ pi,
                  int auto_reset, int words_per_warp) {
  const int wib = threadIdx.x >> 5;
  const int g = blockIdx.x * RZ_TREE_WARPS + wib;
  if (g >= t.n_trees) return;
  const int lane = rz_lane();
  const rz_geom q = rz_geom_of(t.game);
  const int H = t.game.board_size, AS = t.game.action_stride;
  uint32_t* bits = rz_adv_smem + (size_t)wib * 2 * words_per_warp;
  uint32_t* wprefix = bits + words_per_warp;
  int32_t* rmeta = t.root_meta + (size_t)g * RZ_META_STRIDE;
  const int m = moves[g];
  if (m < 0) {  // reset_player(): update_with_move(-1)  (alphazero_mcts.py:132-134)
    if (lane == 0) rz_tree_fresh(t, g, 0, 0.0);
    return;
  }
  if (rmeta[RZ_META_STATUS] != RZ_ACTIVE) return;
  typename GM::board b;
  GM::load_root(b, t, g);
  if (GM::action_illegal(b, m, q)) {  // gomoku_env.py:51 / go_base IllegalMove
    if (lane == 0) rmeta[RZ_META_FAULT] |= RZ_FAULT_ILLEGAL_MOVE;
    return;
  }
  const int ply = rmeta[RZ_META_PLY];
  // game.py:113-115: (current_state, move_probs, current_player) before the move
  if (have_traj) {
    if (ply < traj.max_plies) {
      const size_t so = (size_t)g * traj.max_plies + ply;
      if (lane < H) {
        traj.stage_rows[so * 2 * H + lane] = b.p[0];
        traj.stage_rows[so * 2 * H + H + lane] = b.p[1];
      }
      if (lane == 0) {
        int32_t* si = traj.stage_info + so * 4;
        si[0] = b.player; si[1] = b.last_move; si[2] = m; si[3] = b.stones;
      }
      for (int s = lane; s < AS; s += 32)
        traj.stage_pi[so * AS + s] = pi ? pi[(size_t)g * AS + s] : 0.0f;
    } else if (lane == 0) {
      rmeta[RZ_META_FAULT] |= RZ_FAULT_TRAJ_OVERFLOW;
    }
  }
  // game.py:117: game_env.step(move)
  GM::play(b, m, q);
  int winner;
  const int status = GM::status(b, q, winner);

  // alphazero_mcts.py:96-103
  const bool root_expanded = t.n_nodes[g] > 0;
  const size_t rb = rz_edge_base(t, g, 0);
  const int cn = root_expanded ? t.edge_N[rb + m] : -1;  // -1: move not among the children
  const double cw = (cn > 0) ? t.edge_W[rb + m] : 0.0;
  const int cc = (cn > 0) ? t.edge_child[rb + m] : -1;
  const int co = (cn > 0 && t.edge_O) ? t.edge_O[rb + m] : 0;   // SearchNode.outcome of the child that becomes the root
  if (!keep_subtree || cn < 0) {
    if (lane == 0) rz_tree_fresh(t, g, 0, 0.0);
  } else if (cc < 0) {  // child exists but was never expanded: it keeps its own counts
    if (lane == 0) { rz_tree_fresh(t, g, cn, cw); if (t.root_O) t.root_O[g] = co; }
  } else {
    const int kept = rz_tree_compact(t, g, cc, bits, wprefix, max_carry);
    if (lane == 0) {
      if (kept < 0) {
        rz_tree_fresh(t, g, 0, 0.0);
        rmeta[RZ_META_FAULT] |= RZ_FAULT_CARRY_DROPPED;
      } else {
        t.n_nodes[g] = kept; t.root_N[g] = cn; t.root_W[g] = cw;
        if (t.root_O) t.root_O[g] = co;
      }
    }
  }

  GM::store_root(b, t, g);
  if (lane == 0) {
    GM::store_meta(b, rmeta);
    rmeta[RZ_META_STATUS] = status;
    rmeta[RZ_META_WINNER] = winner;
    rmeta[RZ_META_PLY] = ply + 1;
  }
  if (status == RZ_ACTIVE) return;

  // game.py:121-134: episode over -> z per ply, flush to the ring, reset_player()
  if (have_traj) {
    const int n = min(ply + 1, traj.max_plies);
    unsigned long long start = 0;
    if (lane == 0) {
      start = atomicAdd(traj.ring_cursor, (unsigned long long)n);
      atomicAdd(traj.games_done, 1ull);
      atomicAdd(traj.plies_done, (unsigned long long)(ply + 1));
    }
    start = __shfl_sync(RZ_FULL, start, 0);
    const int episode = rmeta[RZ_META_EPISODE];
    for (int j = 0; j < n; ++j) {
      const size_t so = (size_t)g * traj.max_plies + j;
      const size_t ro = (size_t)((start + j) % (unsigned long long)traj.ring_capacity);
      if (lane < H) {
        traj.ring_rows[ro * 2 * H + lane] = traj.stage_rows[so * 2 * H + lane];
        traj.ring_rows[ro * 2 * H + H + lane] = traj.stage_rows[so * 2 * H + H + lane];
      }
      if (lane == 0) {
        const int mover = traj.stage_info[so * 4 + 0];
        int32_t* ri = traj.ring_info + ro * 6;
        ri[0] = mover;
        ri[1] = traj.stage_info[so * 4 + 1];
        ri[2] = winner < 0 ? 0 : (mover == winner ? 1 : -1);
        ri[3] = g;
        ri[4] = episode;
        ri[5] = j;
      }
      for (int s = lane; s < AS; s += 32) traj.ring_pi[ro * AS + s] = traj.stage_pi[so * AS + s];
    }
  }
  if (lane == 0) rz_tree_fresh(t, g, 0, 0.0);
  if (auto_reset) {
    GM::clear_root(t, g);
    if (lane == 0) {
      rmeta[RZ_META_PLAYER] = 0;
      rmeta[RZ_META_LAST_MOVE] = -1;
      rmeta[RZ_META_STONES] = 0;
      rmeta[RZ_META_STATUS] = RZ_ACTIVE;
      rmeta[RZ_META_WINNER] = -1;
      rmeta[RZ_META_PLY] = 0;
      rmeta[RZ_META_EPISODE] += 1;
    }
  }
}

// ---------------------------------------------------------------------------
// Evaluation match (GameControl.start_play, game.py:61-94) for G games at once: tree g of both seats' forests is
// game g, the mover's root is ACTIVE and the other seat's IDLE.  One warp per game plays the mover's move, hands the
// position over and gives both seats fresh trees (neither player keeps a tree between moves, alphazero_mcts.py:158,
// rollout_mcts.py:131).
// ---------------------------------------------------------------------------
template <class GM>
__global__ void __launch_bounds__(RZ_TREE_THREADS)
rz_match_commit_kernel(rz_tree_desc t0, rz_tree_desc t1, const int32_t* __restrict__ moves0,
                       const int32_t* __restrict__ moves1, int32_t* __restrict__ move_log, int max_plies) {
  const int g = blockIdx.x * RZ_TREE_WARPS + (threadIdx.x >> 5);
  if (g >= t0.n_trees) return;
  const int lane = rz_lane();
  const rz_geom q = rz_geom_of(t0.game);
  int32_t* m0 = t0.root_meta + (size_t)g * RZ_META_STRIDE;
  int32_t* m1 = t1.root_meta + (size_t)g * RZ_META_STRIDE;
  const int seat = m0[RZ_META_STATUS] == RZ_ACTIVE ? 0 : (m1[RZ_META_STATUS] == RZ_ACTIVE ? 1 : -1);
  if (seat < 0) return;                       // game over
  const rz_tree_desc& tm = seat ? t1 : t0;    // the mover's forest
  const rz_tree_desc& to = seat ? t0 : t1;
  int32_t* mm = seat ? m1 : m0;
  int32_t* mo = seat ? m0 : m1;
  const int32_t* moves = seat ? moves1 : moves0;
  if (tm.n_nodes[g] == 0) {                   // no search ran on the mover's root: nothing to choose from
    if (lane == 0) mm[RZ_META_FAULT] |= RZ_FAULT_NO_CHILDREN;
    return;
  }
  int m;
  if (moves) {
    m = moves[g];
  } else {
    // the first most-visited child: max over (N desc, action asc) of the root's children (edge_N >= 0)
    const size_t base = rz_edge_base(tm, g, 0);
    int bn = -1, bs = 0x7fffffff;
    for (int s = lane; s < tm.game.action_stride; s += 32) {
      const int n = tm.edge_N[base + s];
      if (n > bn) { bn = n; bs = s; }           // s ascends per lane: the first maximum of the lane
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int n2 = __shfl_xor_sync(RZ_FULL, bn, o);
      const int s2 = __shfl_xor_sync(RZ_FULL, bs, o);
      if (n2 > bn || (n2 == bn && s2 < bs)) { bn = n2; bs = s2; }
    }
    m = bn >= 0 ? bs : -1;
  }
  typename GM::board b;
  GM::load_root(b, tm, g);
  if (m < 0 || GM::action_illegal(b, m, q)) {
    if (lane == 0) mm[RZ_META_FAULT] |= RZ_FAULT_ILLEGAL_MOVE;
    return;
  }
  const int ply = mm[RZ_META_PLY];
  GM::play(b, m, q);
  int winner;
  const int status = GM::status(b, q, winner);
  // both roots hold the position after the move; only the other seat's is searched next
  GM::store_root(b, to, g);
  GM::store_root(b, tm, g);
  if (lane == 0) {
    if (ply < max_plies) move_log[(size_t)g * max_plies + ply] = m;
    GM::store_meta(b, mo);
    GM::store_meta(b, mm);
    mo[RZ_META_STATUS] = status;
    mm[RZ_META_STATUS] = status == RZ_ACTIVE ? RZ_IDLE : status;
    mo[RZ_META_WINNER] = mm[RZ_META_WINNER] = winner;
    mo[RZ_META_PLY] = mm[RZ_META_PLY] = ply + 1;
    rz_tree_fresh(to, g, 0, 0.0);
    rz_tree_fresh(tm, g, 0, 0.0);
  }
}

// ---------------------------------------------------------------------------
// SearchNode.best_child (deepmind_mcts.py:153-175): max over the root's children of the key
// (outcome[player] or 0, explore_count, total_reward); first maximum wins.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(RZ_TREE_THREADS)
rz_best_child_kernel(rz_tree_desc t, int32_t* __restrict__ best, int32_t* __restrict__ outcome_out) {
  const int g = blockIdx.x * RZ_TREE_WARPS + (threadIdx.x >> 5);
  if (g >= t.n_trees) return;
  const int lane = rz_lane();
  const int AS = t.game.action_stride;
  const int rp = t.root_meta[(size_t)g * RZ_META_STRIDE + RZ_META_PLAYER] & 1;
  const size_t base = rz_edge_base(t, g, 0);
  int bo = -2, bn = -1, bs = 0x7fffffff, br = 0;   // br: position in the (shuffled) children list, 0 if unshuffled
  double bw = 0.0;
  if (t.n_nodes[g] > 0) {
    for (int s = lane; s < AS; s += 32) {
      const int n = t.edge_N[base + s];
      if (n < 0) continue;
      const int c = t.edge_O ? t.edge_O[base + s] : 0;
      const int o = c ? rz_outcome_of(c, rp) : 0;
      const double w = n > 0 ? t.edge_W[base + s] : 0.0;
      const int r = t.edge_R ? t.edge_R[base + s] : 0;
      if (bs == 0x7fffffff || o > bo || (o == bo && (n > bn || (n == bn && (w > bw || (w == bw && r < br)))))) {
        bo = o; bn = n; bw = w; bs = s; br = r;
      }
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const int o2 = __shfl_xor_sync(RZ_FULL, bo, off);
    const int n2 = __shfl_xor_sync(RZ_FULL, bn, off);
    const double w2 = __shfl_xor_sync(RZ_FULL, bw, off);
    const int s2 = __shfl_xor_sync(RZ_FULL, bs, off);
    const int r2 = __shfl_xor_sync(RZ_FULL, br, off);
    if (s2 == 0x7fffffff) continue;
    const bool greater = bs == 0x7fffffff || o2 > bo || (o2 == bo && (n2 > bn || (n2 == bn && w2 > bw)));
    const bool equal = bs != 0x7fffffff && o2 == bo && n2 == bn && w2 == bw;
    if (greater || (equal && (r2 < br || (r2 == br && s2 < bs)))) { bo = o2; bn = n2; bw = w2; bs = s2; br = r2; }
  }
  if (lane == 0) {
    best[g] = bs == 0x7fffffff ? -1 : bs;
    if (outcome_out) outcome_out[g] = t.root_O ? t.root_O[g] : 0;
  }
}

// ---------------------------------------------------------------------------
// Utility kernels + C ABI
// ---------------------------------------------------------------------------
__global__ void rz_tree_reset_kernel(rz_tree_desc t, const uint8_t* __restrict__ mask) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= t.n_trees) return;
  if (mask && !mask[g]) return;
  t.n_nodes[g] = 0;
  t.root_N[g] = 0;
  t.root_W[g] = 0.0;
  t.depth[g] = -1;
  if (t.root_O) t.root_O[g] = 0;
}

static int rz_check_tree(const rz_tree_desc* t, const char* who) {
  RZ_REQUIRE(t, "%s: null tree desc", who);
  if (rz_check_game(&t->game)) return -1;
  RZ_REQUIRE(t->n_trees >= 0, "%s: n_trees %d", who, t->n_trees);
  RZ_REQUIRE(t->max_nodes >= 1, "%s: max_nodes %d", who, t->max_nodes);
  RZ_REQUIRE(t->max_depth >= 1, "%s: max_depth %d", who, t->max_depth);
  RZ_REQUIRE(t->game.action_stride <= 32 * RZ_MAX_ITERS, "%s: action_stride %d > %d", who,
             t->game.action_stride, 32 * RZ_MAX_ITERS);
  RZ_REQUIRE(t->rule == RZ_RULE_UCT || t->rule == RZ_RULE_PUCT, "%s: rule %d", who, t->rule);
  RZ_REQUIRE(t->edge_N && t->edge_W && t->edge_child && t->node_parent && t->node_paction,
             "%s: null node pool", who);
  RZ_REQUIRE(t->rule != RZ_RULE_PUCT || (t->edge_P && t->store_priors),
             "%s: the PUCT rule needs stored priors", who);
  RZ_REQUIRE(!t->store_priors || t->edge_P, "%s: store_priors set but edge_P is null", who);
  RZ_REQUIRE(t->n_nodes && t->root_N && t->root_W && t->root_rows && t->root_meta,
             "%s: null per-tree array", who);
  RZ_REQUIRE(t->path_node && t->path_action && t->depth && t->leaf_rows && t->leaf_meta,
             "%s: null wave scratch", who);
  RZ_REQUIRE(t->ln_table && t->ln_table_len >= 2, "%s: ln table missing", who);
  RZ_REQUIRE(t->game.game_type != RZ_GAME_GO || (t->root_hist && t->leaf_hist),
             "%s: Go needs the root_hist / leaf_hist planes", who);
  RZ_REQUIRE(t->flavour == RZ_FLAVOUR_ALPHAZERO || t->flavour == RZ_FLAVOUR_DEEPMIND, "%s: flavour %d", who, t->flavour);
  RZ_REQUIRE(t->flavour != RZ_FLAVOUR_DEEPMIND || (t->edge_O && t->root_O),
             "%s: the DeepMindMCTS flavour needs the outcome arrays edge_O / root_O", who);
  RZ_REQUIRE(t->returns_mode == RZ_RETURNS_REFERENCE || t->returns_mode == RZ_RETURNS_ZERO_SUM,
             "%s: returns_mode %d", who, t->returns_mode);
  RZ_REQUIRE(t->leaves_per_tree >= 0 && t->leaves_per_tree <= 256, "%s: leaves_per_tree %d outside [0,256]", who,
             t->leaves_per_tree);
  RZ_REQUIRE(!t->edge_P64 || t->store_priors, "%s: edge_P64 needs store_priors", who);
  RZ_REQUIRE(!t->edge_R || t->flavour == RZ_FLAVOUR_DEEPMIND, "%s: edge_R (child shuffle) belongs to the DeepMindMCTS flavour", who);
  RZ_REQUIRE(t->shuffle_mode == 0 || t->shuffle_mode == 1, "%s: shuffle_mode %d", who, t->shuffle_mode);
  if (t->leaves_per_tree > 1) {
    RZ_REQUIRE(t->flavour == RZ_FLAVOUR_ALPHAZERO, "%s: leaf-parallel waves (leaves_per_tree %d) need the AlphaZero flavour",
               who, t->leaves_per_tree);
    RZ_REQUIRE(t->vl_saved_W, "%s: leaves_per_tree %d needs the vl_saved_W scratch", who, t->leaves_per_tree);
    RZ_REQUIRE(t->virtual_loss >= 0.0, "%s: virtual_loss %f", who, t->virtual_loss);
  }
  return 0;
}

static inline dim3 rz_tree_grid(int n) { return dim3((unsigned)((n + RZ_TREE_WARPS - 1) / RZ_TREE_WARPS)); }

extern "C" int rz_tree_reset(const rz_tree_desc* t, const uint8_t* tree_mask, void* stream) {
  if (rz_check_tree(t, "rz_tree_reset")) return -1;
  if (t->n_trees == 0) return 0;
  rz_tree_reset_kernel<<<(t->n_trees + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*t, tree_mask);
  RZ_LAUNCH_CHECK("rz_tree_reset");
  return 0;
}

extern "C" int rz_tree_select(const rz_tree_desc* t, void* stream) {
  if (rz_check_tree(t, "rz_tree_select")) return -1;
  if (t->n_trees == 0) return 0;
  const dim3 grid = rz_tree_grid(t->n_trees);
  cudaStream_t st = (cudaStream_t)stream;
  const bool go = t->game.game_type == RZ_GAME_GO, dm = t->flavour == RZ_FLAVOUR_DEEPMIND;
  if (go && dm) rz_launch_pdl(rz_select_kernel<rz_go_game, true>, grid, RZ_TREE_THREADS, 0, st, *t);
  else if (go) rz_launch_pdl(rz_select_kernel<rz_go_game, false>, grid, RZ_TREE_THREADS, 0, st, *t);
  else if (dm) rz_launch_pdl(rz_select_kernel<rz_line_game, true>, grid, RZ_TREE_THREADS, 0, st, *t);
  else rz_launch_pdl(rz_select_kernel<rz_line_game, false>, grid, RZ_TREE_THREADS, 0, st, *t);
  RZ_LAUNCH_CHECK("rz_tree_select");
  return 0;
}

static int rz_expand_backup_launch(const rz_tree_desc* t, const float* prior, int prior_is_log,
                                   const float* value, const double* value64, float noise_eps,
                                   float noise_alpha, unsigned long long seed, void* stream,
                                   const double* noise64 = nullptr, const double* prior64 = nullptr);

extern "C" int rz_tree_expand_backup_dm(const rz_tree_desc* t, const float* prior, int prior_is_log,
                                        const float* value, const double* ret64, float noise_eps,
                                        float noise_alpha, unsigned long long seed, void* stream) {
  if (rz_check_tree(t, "rz_tree_expand_backup_dm")) return -1;
  RZ_REQUIRE(t->flavour == RZ_FLAVOUR_DEEPMIND, "rz_tree_expand_backup_dm: the tree is not in the DeepMindMCTS flavour");
  return rz_expand_backup_launch(t, prior, prior_is_log, value, ret64, noise_eps, noise_alpha, seed, stream);
}

extern "C" int rz_tree_expand_backup(const rz_tree_desc* t, const float* prior, int prior_is_log,
                                     const float* value, const double* value64, float noise_eps,
                                     float noise_alpha,
                                     unsigned long long seed, void* stream) {
  if (rz_check_tree(t, "rz_tree_expand_backup")) return -1;
  RZ_REQUIRE(t->flavour == RZ_FLAVOUR_ALPHAZERO, "rz_tree_expand_backup: DeepMindMCTS trees use rz_tree_expand_backup_dm");
  return rz_expand_backup_launch(t, prior, prior_is_log, value, value64, noise_eps, noise_alpha, seed, stream);
}

extern "C" int rz_tree_expand_backup_ex(const rz_tree_desc* t, const float* prior, int prior_is_log,
                                        const float* value, const double* value64, float noise_eps,
                                        float noise_alpha, unsigned long long seed, const double* noise64,
                                        const double* prior64, void* stream) {
  if (rz_check_tree(t, "rz_tree_expand_backup_ex")) return -1;
  RZ_REQUIRE(!(noise64 && prior64), "rz_tree_expand_backup_ex: give noise64 or prior64, not both");
  RZ_REQUIRE(!noise64 || (noise_eps > 0.0f && prior), "rz_tree_expand_backup_ex: noise64 needs noise_eps > 0 and a prior");
  return rz_expand_backup_launch(t, prior, prior_is_log, value, value64, noise_eps, noise_alpha, seed, stream, noise64,
                                 prior64);
}

extern "C" int rz_tree_expand_backup_select(const rz_tree_desc* t, const float* prior, int prior_is_log,
                                            const float* value, const double* value64, float noise_eps,
                                            float noise_alpha, unsigned long long seed, void* stream) {
  if (rz_check_tree(t, "rz_tree_expand_backup_select")) return -1;
  RZ_REQUIRE(t->leaves_per_tree <= 1, "rz_tree_expand_backup_select: one leaf per tree and wave only (leaves_per_tree %d)",
             t->leaves_per_tree);
  RZ_REQUIRE(value || value64, "rz_tree_expand_backup_select: null value");
  RZ_REQUIRE(prior || !t->store_priors, "rz_tree_expand_backup_select: null prior with store_priors");
  RZ_REQUIRE(noise_eps >= 0.0f && noise_eps <= 1.0f, "rz_tree_expand_backup_select: noise_eps %f", noise_eps);
  RZ_REQUIRE(noise_eps == 0.0f || noise_alpha > 0.0f, "rz_tree_expand_backup_select: noise_alpha %f", noise_alpha);
  if (t->n_trees == 0) return 0;
  const dim3 grid = rz_tree_grid(t->n_trees);
  cudaStream_t st = (cudaStream_t)stream;
  const bool go = t->game.game_type == RZ_GAME_GO, dm = t->flavour == RZ_FLAVOUR_DEEPMIND;
#define RZ_EBS_ARGS *t, prior, prior_is_log, value, value64, noise_eps, noise_alpha, seed, t->global_offset
  if (go && dm) rz_launch_pdl(rz_expand_backup_select_kernel<rz_go_game, true>, grid, RZ_TREE_THREADS, 0, st, RZ_EBS_ARGS);
  else if (go) rz_launch_pdl(rz_expand_backup_select_kernel<rz_go_game, false>, grid, RZ_TREE_THREADS, 0, st, RZ_EBS_ARGS);
  else if (dm) rz_launch_pdl(rz_expand_backup_select_kernel<rz_line_game, true>, grid, RZ_TREE_THREADS, 0, st, RZ_EBS_ARGS);
  else rz_launch_pdl(rz_expand_backup_select_kernel<rz_line_game, false>, grid, RZ_TREE_THREADS, 0, st, RZ_EBS_ARGS);
#undef RZ_EBS_ARGS
  RZ_LAUNCH_CHECK("rz_tree_expand_backup_select");
  return 0;
}

static int rz_expand_backup_launch(const rz_tree_desc* t, const float* prior, int prior_is_log,
                                   const float* value, const double* value64, float noise_eps,
                                   float noise_alpha, unsigned long long seed, void* stream,
                                   const double* noise64, const double* prior64) {
  RZ_REQUIRE(value || value64, "rz_tree_expand_backup: null value");
  RZ_REQUIRE(prior || prior64 || !t->store_priors, "rz_tree_expand_backup: null prior with store_priors");
  RZ_REQUIRE(noise_eps >= 0.0f && noise_eps <= 1.0f, "rz_tree_expand_backup: noise_eps %f", noise_eps);
  RZ_REQUIRE(noise_eps == 0.0f || noise_alpha > 0.0f, "rz_tree_expand_backup: noise_alpha %f", noise_alpha);
  if (t->n_trees == 0) return 0;
  const dim3 grid = rz_tree_grid(t->n_trees);
  cudaStream_t st = (cudaStream_t)stream;
  const bool go = t->game.game_type == RZ_GAME_GO, dm = t->flavour == RZ_FLAVOUR_DEEPMIND;
#define RZ_EB_ARGS *t, prior, prior_is_log, value, value64, noise_eps, noise_alpha, seed, t->global_offset, noise64, prior64
  if (go && dm) rz_launch_pdl(rz_expand_backup_kernel<rz_go_game, true>, grid, RZ_TREE_THREADS, 0, st, RZ_EB_ARGS);
  else if (go) rz_launch_pdl(rz_expand_backup_kernel<rz_go_game, false>, grid, RZ_TREE_THREADS, 0, st, RZ_EB_ARGS);
  else if (dm) rz_launch_pdl(rz_expand_backup_kernel<rz_line_game, true>, grid, RZ_TREE_THREADS, 0, st, RZ_EB_ARGS);
  else rz_launch_pdl(rz_expand_backup_kernel<rz_line_game, false>, grid, RZ_TREE_THREADS, 0, st, RZ_EB_ARGS);
#undef RZ_EB_ARGS
  RZ_LAUNCH_CHECK("rz_tree_expand_backup");
  return 0;
}

extern "C" int rz_tree_root_policy(const rz_tree_desc* t, double temperature, int32_t* visits,
                                   float* pi, int32_t* move, const double* u01,
                                   unsigned long long seed, void* stream) {
  if (rz_check_tree(t, "rz_tree_root_policy")) return -1;
  RZ_REQUIRE(temperature > 0.0, "rz_tree_root_policy: temperature %g", temperature);
  if (t->n_trees == 0) return 0;
  rz_root_policy_kernel<<<rz_tree_grid(t->n_trees), RZ_TREE_THREADS, 0, (cudaStream_t)stream>>>(
      *t, temperature, visits, pi, move, u01, seed, t->global_offset);
  RZ_LAUNCH_CHECK("rz_tree_root_policy");
  return 0;
}

extern "C" int rz_tree_advance(const rz_tree_desc* t, const int32_t* moves, int keep_subtree,
                               int max_carry, const rz_traj_desc* traj, const float* pi,
                               int auto_reset, void* stream) {
  if (rz_check_tree(t, "rz_tree_advance")) return -1;
  RZ_REQUIRE(moves, "rz_tree_advance: null moves");
  RZ_REQUIRE(max_carry >= 0 && max_carry <= t->max_nodes, "rz_tree_advance: max_carry %d", max_carry);
  rz_traj_desc td;
  memset(&td, 0, sizeof(td));
  if (traj) {
    td = *traj;
    RZ_REQUIRE(td.max_plies >= 1 && td.ring_capacity >= td.max_plies, "rz_tree_advance: trajectory sizes");
    RZ_REQUIRE(td.stage_rows && td.stage_info && td.stage_pi && td.ring_rows && td.ring_info &&
                   td.ring_pi && td.ring_cursor && td.games_done && td.plies_done,
               "rz_tree_advance: null trajectory buffer");
  }
  if (t->n_trees == 0) return 0;
  const int words = (t->max_nodes + 31) / 32;
  const size_t smem = (size_t)RZ_TREE_WARPS * 2 * words * sizeof(uint32_t);
  RZ_REQUIRE(smem <= 48 * 1024, "rz_tree_advance: max_nodes %d needs %zu B of shared memory", t->max_nodes, smem);
  if (t->game.game_type == RZ_GAME_GO)
    rz_advance_kernel<rz_go_game><<<rz_tree_grid(t->n_trees), RZ_TREE_THREADS, smem, (cudaStream_t)stream>>>(
        *t, moves, keep_subtree, max_carry, td, traj != nullptr, pi, auto_reset, words);
  else
    rz_advance_kernel<rz_line_game><<<rz_tree_grid(t->n_trees), RZ_TREE_THREADS, smem, (cudaStream_t)stream>>>(
        *t, moves, keep_subtree, max_carry, td, traj != nullptr, pi, auto_reset, words);
  RZ_LAUNCH_CHECK("rz_tree_advance");
  return 0;
}

extern "C" int rz_match_commit(const rz_tree_desc* seat0, const rz_tree_desc* seat1, const int32_t* moves0,
                               const int32_t* moves1, int32_t* move_log, int max_plies, void* stream) {
  if (rz_check_tree(seat0, "rz_match_commit (seat 0)") || rz_check_tree(seat1, "rz_match_commit (seat 1)")) return -1;
  RZ_REQUIRE(memcmp(&seat0->game, &seat1->game, sizeof(rz_game_desc)) == 0,
             "rz_match_commit: the seats' game descriptors differ");
  RZ_REQUIRE(seat0->n_trees == seat1->n_trees, "rz_match_commit: n_trees %d vs %d", seat0->n_trees, seat1->n_trees);
  RZ_REQUIRE(seat0->game.game_type != RZ_GAME_GO, "rz_match_commit: Go is not supported");
  RZ_REQUIRE(seat0->flavour == RZ_FLAVOUR_ALPHAZERO && seat1->flavour == RZ_FLAVOUR_ALPHAZERO,
             "rz_match_commit: the DeepMindMCTS flavour is not supported");
  RZ_REQUIRE(seat0->leaves_per_tree <= 1 && seat1->leaves_per_tree <= 1,
             "rz_match_commit: leaves_per_tree %d / %d (one leaf per wave only)", seat0->leaves_per_tree,
             seat1->leaves_per_tree);
  RZ_REQUIRE(move_log, "rz_match_commit: null move_log");
  const int W = seat0->game.width > 0 ? seat0->game.width : seat0->game.board_size;
  RZ_REQUIRE(max_plies >= seat0->game.board_size * W, "rz_match_commit: max_plies %d below the board's %d cells",
             max_plies, seat0->game.board_size * W);
  if (seat0->n_trees == 0) return 0;
  rz_match_commit_kernel<rz_line_game><<<rz_tree_grid(seat0->n_trees), RZ_TREE_THREADS, 0, (cudaStream_t)stream>>>(
      *seat0, *seat1, moves0, moves1, move_log, max_plies);
  RZ_LAUNCH_CHECK("rz_match_commit");
  return 0;
}

extern "C" int rz_tree_best_child(const rz_tree_desc* t, int32_t* best, int32_t* outcome_out, void* stream) {
  if (rz_check_tree(t, "rz_tree_best_child")) return -1;
  RZ_REQUIRE(best, "rz_tree_best_child: null output");
  if (t->n_trees == 0) return 0;
  rz_best_child_kernel<<<rz_tree_grid(t->n_trees), RZ_TREE_THREADS, 0, (cudaStream_t)stream>>>(*t, best, outcome_out);
  RZ_LAUNCH_CHECK("rz_tree_best_child");
  return 0;
}
