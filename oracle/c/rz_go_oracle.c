/* TEST INFRASTRUCTURE ONLY -- plain-C restatement of the Go rules and of the AlphaZero search over them, so that a
 * full BASELINE-size batch (8192 trees x 800 playouts on 19x19, config 4) can be checked tree by tree in seconds.
 * PARITY UNPINNED against the reference: its Go engine is pettingzoo.classic.go.go_base (third party, absent); this
 * file restates oracle/go_oracle.py (itself the published MiniGo algorithm at the reference's call sites,
 * rlzero/games/go/go_env.py:98-112,168-210) a second time and is pinned to it on the CPU by tests/test_go_oracle_c.py
 * (random games: boards, ko, legal masks, scores; searches: visit counts and value sums bit for bit).
 *
 * Rules: capture of liberty-less opponent groups, no suicide, simple ko, pass = action N*N, two consecutive passes end
 * the game, Tromp-Taylor area score minus komi; player 0 = black moves first.  Search: rlzero/mcts/alphazero_mcts.py
 * :42-71 + node.py:32-144 exactly as oracle/c/rz_oracle.c plays it for the line games (UCB1 of the reference, or the
 * PUCT formula of deepmind_mcts.py:149-151), children keyed by ascending action, first maximum wins, the evaluator is
 * called on terminal leaves too, leaf value from the side to move, sign flipped per level.
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (oracle/build_oracle.py). */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define GMAX 361

typedef struct {
  int N;
  int8_t cell[GMAX];      /* 0 empty, +1 black, -1 white */
  int ko;                 /* square that may not be retaken, -1 none */
  int to_play;            /* +1 black, -1 white */
  int n;                  /* moves played (Position.n) */
  int pass1, pass2;       /* the last / the one before last move was a pass */
  int last_action;        /* -1 before the first move; N*N for a pass */
  double komi;
  int max_moves;
} gob_t;

static void gob_reset(gob_t* b, int N, double komi, int max_moves) {
  memset(b, 0, sizeof(*b));
  b->N = N; b->ko = -1; b->to_play = 1; b->last_action = -1; b->komi = komi; b->max_moves = max_moves;
}

static int nbrs(int N, int c, int* out) {
  const int r = c / N, w = c % N;
  int k = 0;
  if (r + 1 < N) out[k++] = c + N;
  if (r > 0) out[k++] = c - N;
  if (w + 1 < N) out[k++] = c + 1;
  if (w > 0) out[k++] = c - 1;
  return k;
}

/* flood the same-colour region of `start`; marks mark[] with `tag`; returns the number of distinct EMPTY points
 * bordering it (its liberties if it is a chain of stones); border colours seen are OR-ed into *colors (1 black, 2 white,
 * 4 empty) */
static int flood(const gob_t* b, int start, int* mark, int tag, int* chain, int* n_chain, int* colors) {
  const int N = b->N, color = b->cell[start];
  int stack[GMAX], sp = 0, libs = 0, nc = 0;
  static __thread int libmark[GMAX];
  static __thread int libtag = 0;
  ++libtag;
  stack[sp++] = start; mark[start] = tag;
  while (sp) {
    const int c = stack[--sp];
    if (chain) chain[nc] = c;
    ++nc;
    int nb[4];
    const int k = nbrs(N, c, nb);
    for (int i = 0; i < k; ++i) {
      const int q = nb[i];
      if (b->cell[q] == color) {
        if (mark[q] != tag) { mark[q] = tag; stack[sp++] = q; }
      } else {
        if (colors) *colors |= b->cell[q] == 1 ? 1 : (b->cell[q] == -1 ? 2 : 4);
        if (b->cell[q] == 0 && libmark[q] != libtag) { libmark[q] = libtag; ++libs; }
      }
    }
  }
  if (n_chain) *n_chain = nc;
  return libs;
}

static __thread int g_mark[GMAX];
static __thread int g_tag = 0;

/* Position.is_move_suicidal */
static int go_suicidal(const gob_t* b, int move) {
  int nb[4];
  const int k = nbrs(b->N, move, nb);
  /* the union of the liberties of the friendly neighbour chains, minus the move itself */
  static __thread int lm[GMAX];
  static __thread int lt = 0;
  ++lt;
  int potential = 0;
  for (int i = 0; i < k; ++i) {
    const int q = nb[i];
    if (b->cell[q] == 0) return 0;                         /* a liberty of its own */
    int chain[GMAX], nc;
    const int libs = flood(b, q, g_mark, ++g_tag, chain, &nc, NULL);
    if (b->cell[q] == b->to_play) {
      /* collect this chain's liberties */
      for (int j = 0; j < nc; ++j) {
        int nb2[4];
        const int k2 = nbrs(b->N, chain[j], nb2);
        for (int t = 0; t < k2; ++t)
          if (b->cell[nb2[t]] == 0 && nb2[t] != move && lm[nb2[t]] != lt) { lm[nb2[t]] = lt; ++potential; }
      }
    } else if (libs == 1) {
      return 0;                                            /* captures that opponent group */
    }
  }
  return potential == 0;
}

static int go_legal(const gob_t* b, int a) {
  if (a == b->N * b->N) return 1;
  if (b->cell[a] != 0) return 0;
  if (a == b->ko) return 0;
  return !go_suicidal(b, a);
}

/* is_koish: colour surrounding the empty point on every side, else 0 */
static int go_koish(const gob_t* b, int c) {
  if (b->cell[c] != 0) return 0;
  int nb[4];
  const int k = nbrs(b->N, c, nb);
  int col = 0;
  for (int i = 0; i < k; ++i) {
    if (b->cell[nb[i]] == 0) return 0;
    if (col == 0) col = b->cell[nb[i]];
    else if (col != b->cell[nb[i]]) return 0;
  }
  return col;
}

/* Position.play_move; returns 0, or -1 if illegal */
static int go_play(gob_t* b, int a) {
  const int NN = b->N * b->N;
  if (a == NN) {
    b->n += 1; b->pass2 = b->pass1; b->pass1 = 1; b->to_play = -b->to_play; b->ko = -1; b->last_action = a;
    return 0;
  }
  if (a < 0 || a > NN || !go_legal(b, a)) return -1;
  const int color = b->to_play;
  const int potential_ko = go_koish(b, a);
  b->cell[a] = (int8_t)color;
  int nb[4];
  const int k = nbrs(b->N, a, nb);
  int captured = 0, cap_sq = -1;
  for (int i = 0; i < k; ++i) {
    const int q = nb[i];
    if (b->cell[q] != -color) continue;
    int chain[GMAX], nc;
    const int libs = flood(b, q, g_mark, ++g_tag, chain, &nc, NULL);
    if (libs == 0) {
      for (int j = 0; j < nc; ++j) b->cell[chain[j]] = 0;
      captured += nc; cap_sq = chain[0];
    }
  }
  b->ko = (captured == 1 && potential_ko == -color) ? cap_sq : -1;
  b->n += 1; b->pass2 = b->pass1; b->pass1 = 0; b->to_play = -color; b->last_action = a;
  return 0;
}

static int go_over(const gob_t* b) { return (b->pass1 && b->pass2) || (b->max_moves > 0 && b->n >= b->max_moves); }

/* Position.score(): Tromp-Taylor area from black's point of view, komi subtracted */
static double go_score(const gob_t* b) {
  const int NN = b->N * b->N;
  int black = 0, white = 0;
  int mark[GMAX];
  memset(mark, 0, sizeof(mark));
  for (int c = 0; c < NN; ++c) {
    if (b->cell[c] == 1) ++black;
    else if (b->cell[c] == -1) ++white;
    else if (mark[c] == 0) {
      int colors = 0, nc = 0;
      flood(b, c, mark, 1, NULL, &nc, &colors);
      if ((colors & 3) == 1) black += nc;
      else if ((colors & 3) == 2) white += nc;
    }
  }
  return (double)(black - white) - b->komi;
}
static int go_result(const gob_t* b) { const double s = go_score(b); return s > 0 ? 1 : (s < 0 ? -1 : 0); }
/* GoSearchBoard.game_end_winner (go_env.py:142-143): black (player 0) iff result() == 1 */
static int go_winner(const gob_t* b) { return go_result(b) == 1 ? 0 : 1; }
static int go_player(const gob_t* b) { return b->to_play == 1 ? 0 : 1; }

/* ---- closed-form evaluators (oracle/evaluators.py) over GoSearchBoard.states / last_move ------------------------- */
static uint32_t go_hash(const gob_t* b) {
  uint32_t h = 0;
  for (int m = 0; m < b->N * b->N; ++m)
    if (b->cell[m]) h += (uint32_t)(m + 1) * (uint32_t)(m + 1) * (3u + 4u * (b->cell[m] == 1 ? 0u : 1u));
  h += 7u * (uint32_t)(b->last_action + 1);
  return h * 2654435761u;
}
static int go_stones(const gob_t* b) { int n = 0; for (int m = 0; m < b->N * b->N; ++m) n += b->cell[m] != 0; return n; }
static double go_eval_value(const gob_t* b, int eval_id) {
  if (eval_id == 1) return (double)((17 * go_stones(b) + 31 * (b->last_action + 1)) % 13 - 6) / 8.0;
  if (eval_id == 2) return (double)((int)((go_hash(b) >> 16) % 129u) - 64) / 64.0;
  return 0.0;
}
static double go_eval_prior(int eval_id, int action, int n_legal, uint32_t h) {
  if (eval_id == 2) return (double)(((uint32_t)action * 29u + (h >> 8)) % 32u + 1u) / 256.0;
  return (double)(1.0f / (float)n_legal);
}

/* ---- search ------------------------------------------------------------------------------------------------------ */
typedef struct gnode_s {
  struct gnode_s* parent;
  struct gnode_s** child;
  int expanded, n;
  double w, prior;
} gnode_t;

typedef struct { char* base; size_t used, cap; } garena_t;
static void* ga_alloc(garena_t* a, size_t sz) {
  sz = (sz + 15) & ~(size_t)15;
  if (a->used + sz > a->cap) {
    size_t nc = a->cap * 2 + sz;
    char* nb = (char*)malloc(nc + 16);
    if (!nb) return NULL;
    *(char**)nb = a->base;
    a->base = nb; a->used = 16; a->cap = nc + 16;
  }
  void* p = a->base + a->used;
  a->used += sz;
  return p;
}
static void ga_free(garena_t* a) { char* b = a->base; while (b) { char* nx = *(char**)b; free(b); b = nx; } a->base = NULL; }
static int ga_init(garena_t* a, size_t cap) {
  a->base = (char*)malloc(cap + 16);
  if (!a->base) return -1;
  *(char**)a->base = NULL; a->used = 16; a->cap = cap + 16;
  return 0;
}

static double gnode_score(const gnode_t* c, double cpuct, int rule) {
  if (rule == 1)
    return (c->n ? c->w / (double)c->n : 0.0) + cpuct * c->prior * sqrt((double)c->parent->n) / (double)(c->n + 1);
  if (c->parent->n == 0 || c->n == 0) return INFINITY;
  return c->w / (double)c->n + cpuct * sqrt(log((double)c->parent->n) / (double)c->n);
}

static int go_playout(garena_t* ar, gnode_t* root, gob_t b, double cpuct, int rule, int eval_id) {
  const int A = b.N * b.N + 1;
  gnode_t* node = root;
  while (node->expanded) {
    int best_a = -1; double best_s = 0.0;
    for (int a = 0; a < A; ++a) {
      gnode_t* c = node->child[a];
      if (!c) continue;
      const double s = gnode_score(c, cpuct, rule);
      if (best_a < 0 || s > best_s) { best_a = a; best_s = s; }
    }
    if (best_a < 0) return -2;
    node = node->child[best_a];
    if (go_play(&b, best_a)) return -5;
  }
  double v = go_eval_value(&b, eval_id);
  if (!go_over(&b)) {
    node->child = (gnode_t**)ga_alloc(ar, sizeof(gnode_t*) * (size_t)A);
    if (!node->child) return -1;
    int legal[GMAX + 1], n_legal = 0;
    for (int a = 0; a < A; ++a) { legal[a] = go_legal(&b, a); n_legal += legal[a]; }
    const uint32_t h = eval_id == 2 ? go_hash(&b) : 0u;
    for (int a = 0; a < A; ++a) {
      node->child[a] = NULL;
      if (!legal[a]) continue;
      gnode_t* c = (gnode_t*)ga_alloc(ar, sizeof(gnode_t));
      if (!c) return -1;
      c->parent = node; c->child = NULL; c->expanded = 0; c->n = 0; c->w = 0.0;
      c->prior = go_eval_prior(eval_id, a, n_legal, h);
      node->child[a] = c;
    }
    node->expanded = 1;
  } else {
    v = go_winner(&b) == go_player(&b) ? 1.0 : -1.0;
  }
  v = -v;
  for (gnode_t* p = node; p; p = p->parent) { p->n += 1; p->w += v; v = -v; }
  return 0;
}

/* G independent searches from the positions reached by moves[g][0..n_moves[g]) (row stride max_moves_in):
 * visits / w [G][N*N+1], root_n / root_w [G]; rc[g] per game (0 ok).  OpenMP over games. */
int rzo_go_search_batch(int G, int N, double komi, int move_cap, const int32_t* moves, const int32_t* n_moves,
                        int max_moves_in, int n_playout, double cpuct, int rule, int eval_id, int32_t* visits, double* w,
                        int32_t* root_n, double* root_w) {
  if (N < 1 || N * N > GMAX) return -3;
  const int A = N * N + 1;
  int bad = 0;
#pragma omp parallel for schedule(dynamic, 8)
  for (int g = 0; g < G; ++g) {
    gob_t b;
    gob_reset(&b, N, komi, move_cap);
    int rc = 0;
    for (int i = 0; i < n_moves[g] && rc == 0; ++i) rc = go_play(&b, moves[(size_t)g * max_moves_in + i]);
    garena_t ar;
    if (rc == 0 && ga_init(&ar, (size_t)1 << 21)) rc = -1;
    if (rc == 0) {
      gnode_t* root = (gnode_t*)ga_alloc(&ar, sizeof(gnode_t));
      memset(root, 0, sizeof(*root));
      root->prior = 1.0;
      for (int i = 0; i < n_playout && rc == 0; ++i) rc = go_playout(&ar, root, b, cpuct, rule, eval_id);
      for (int a = 0; a < A; ++a) {
        gnode_t* c = root->expanded ? root->child[a] : NULL;
        visits[(size_t)g * A + a] = c ? c->n : 0;
        w[(size_t)g * A + a] = c ? c->w : 0.0;
      }
      root_n[g] = root->n; root_w[g] = root->w;
      ga_free(&ar);
    }
    if (rc) {
#pragma omp atomic write
      bad = rc;
    }
  }
  return bad;
}

/* Random legal games by the oracle's own rules: game g plays uniformly random legal moves (the pass with probability
 * about 1/32 while other moves exist) from a xorshift stream seeded by (seed, g), at most n_plies[g] of them, stopping
 * at the end of the game.  Outputs the moves [G][max_plies] (-1 padded) and, after the last move, the position: cell
 * [G][N*N] (0 / +1 / -1), ko, to_play (0 black / 1 white), over, score (float64), legal mask [G][N*N+1]. */
int rzo_go_random_games(int G, int N, double komi, int move_cap, const int32_t* n_plies, int max_plies, uint64_t seed,
                        int32_t* moves, int32_t* played, int8_t* cell, int32_t* ko, int32_t* to_play, int32_t* over,
                        double* score, int8_t* legal_out) {
  if (N < 1 || N * N > GMAX) return -3;
  const int NN = N * N, A = NN + 1;
#pragma omp parallel for schedule(dynamic, 8)
  for (int g = 0; g < G; ++g) {
    uint64_t s = seed * 0x9E3779B97F4A7C15ull + (uint64_t)(g + 1) * 0xD1B54A32D192ED03ull;
    gob_t b;
    gob_reset(&b, N, komi, move_cap);
    int k = 0;
    for (; k < n_plies[g] && k < max_plies && !go_over(&b); ++k) {
      int legal[GMAX + 1], n_legal = 0;
      for (int a = 0; a < NN; ++a) { legal[a] = go_legal(&b, a); n_legal += legal[a]; }
      s ^= s << 13; s ^= s >> 7; s ^= s << 17;
      int a = NN;
      if (n_legal > 0 && (s >> 40) % 32u != 0u) {
        int pick = (int)((s >> 8) % (uint64_t)n_legal);
        for (a = 0; a < NN; ++a) if (legal[a] && pick-- == 0) break;
      }
      go_play(&b, a);
      moves[(size_t)g * max_plies + k] = a;
    }
    played[g] = k;
    for (int i = k; i < max_plies; ++i) moves[(size_t)g * max_plies + i] = -1;
    for (int c = 0; c < NN; ++c) cell[(size_t)g * NN + c] = b.cell[c];
    ko[g] = b.ko; to_play[g] = go_player(&b); over[g] = go_over(&b); score[g] = go_score(&b);
    for (int a = 0; a < A; ++a) legal_out[(size_t)g * A + a] = (int8_t)(go_over(&b) ? a == NN : go_legal(&b, a));
  }
  return 0;
}

/* ---- the device's random playouts (rz_eval_rollout_dm_kernel<rz_go_game>, rlzero_b200/csrc/rz_game.cu:342-389) ------
 * Philox-4x32-10 as rz_philox4 (rz_common.cuh:178-195); oracle/philox.py restates it in Python and the CPU tests pin
 * both to the Random123 known-answer vectors. */
static void rzo_philox4_(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t out[4]) {
  uint32_t c[4] = {c0, c1, c2, c3};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1,
                   n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

void rzo_philox4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t* out) {
  rzo_philox4_(c0, c1, c2, c3, seed, out);
}

/* mean returns of n_rollouts random playouts from one position (cell[N*N] +1 / -1 / 0, to_play +1 black / -1 white,
 * n moves played, pass1 / pass2 = the last / the one before last move was a pass).  Playout r, ply i: counter
 * (g, visit, r << 16 | i, 0xd311); the candidates are the legal points ascending, then the pass; the status is tested
 * before every move and once more after n_limit moves, a playout cut there returns [0, 0].  out[2] = sum / n_rollouts
 * for (black, white); legal_out[N*N + 1] = the legal mask of the position (the evaluator's priors). */
int rzo_go_rollout_dm(int N, double komi, int max_moves, const int8_t* cell, int ko, int to_play, int n, int pass1,
                      int pass2, int n_rollouts, int n_limit, uint32_t g, uint32_t visit, uint64_t seed, double* out,
                      int8_t* legal_out) {
  if (N < 1 || N * N > GMAX || n_rollouts < 1 || n_limit < 0) return -3;
  const int NN = N * N;
  gob_t b0;
  gob_reset(&b0, N, komi, max_moves);
  for (int c = 0; c < NN; ++c) b0.cell[c] = cell[c];
  b0.ko = ko; b0.to_play = to_play; b0.n = n; b0.pass1 = pass1; b0.pass2 = pass2;
  for (int a = 0; a <= NN; ++a) legal_out[a] = (int8_t)go_legal(&b0, a);
  int sum0 = 0, sum1 = 0;
  for (int r = 0; r < n_rollouts; ++r) {
    gob_t b = b0;
    for (int i = 0; i <= n_limit; ++i) {
      if (go_over(&b) || i == n_limit) break;
      int cand[GMAX + 1], n_act = 0;
      for (int a = 0; a < NN; ++a) if (go_legal(&b, a)) cand[n_act++] = a;
      cand[n_act++] = NN;                                  /* the pass is the last candidate */
      uint32_t w[4];
      rzo_philox4_(g, visit, ((uint32_t)r << 16) | (uint32_t)i, 0xd311u, seed, w);
      const int pick = (int)(((uint64_t)w[0] * (uint64_t)n_act) >> 32);
      if (go_play(&b, cand[pick]) != 0) return -4;
    }
    if (go_over(&b)) {                                     /* rz_game_returns: Go always ends decided */
      const int r0 = go_winner(&b) == 0 ? 1 : -1;
      sum0 += r0; sum1 -= r0;
    }
  }
  out[0] = (double)sum0 / (double)n_rollouts;
  out[1] = (double)sum1 / (double)n_rollouts;
  return 0;
}
