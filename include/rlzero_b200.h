/* rlzero_b200 -- C ABI of the B200-native batched self-play MCTS hot path.
 *
 * The reference (jianzhnie/RLZero) has no FFI layer; its boundary is the
 * duck-typed Python API of rlzero/mcts/alphazero_mcts.py and
 * rlzero/games/gomoku/ (SURVEY.md section 8b).  This header is the C-ABI a
 * maintainer would bind underneath those classes (ctypes stub in
 * INTEGRATION.md).  Each entry point cites the reference function it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless it is marked
 *     "host"; the library allocates nothing and keeps no global state except
 *     the last-error string;
 *   - every call is asynchronous on the cudaStream_t passed as `stream`
 *     (void* so that this header needs no CUDA include), performs no host
 *     synchronisation and is CUDA-graph capturable;
 *   - return value 0 = launched, <0 = argument/launch error (rz_last_error()).
 *     Data-dependent faults (illegal move, pool overflow) are reported through
 *     the per-game `fault` words, which the host shim turns into the
 *     reference's exceptions (AssertionError illegal move gomoku_env.py:51,
 *     ValueError('Node has no children.') node.py:39).
 *
 * Layouts
 *   board      : per game 2 x H uint32 row bitmasks, rows[g][c][r] bit w set <=>
 *                stone of player c on square r*W+w  (gomoku_env.py: states dict);
 *                meta last_move holds the SQUARE of the last stone (== the action for Gomoku)
 *   meta       : per game RZ_META_STRIDE int32 (enum rz_meta)
 *   edge block : per expanded node A slots indexed BY ACTION (slot a <=> child
 *                reached by move a; children of a reference node are keyed by
 *                action in ascending order, node.py:71-73), padded to
 *                AS = round_up(A,32):  N int32 (-1 = illegal/no child),
 *                W float64, P float32, child int32.
 */
#ifndef RLZERO_B200_H
#define RLZERO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RZ_ABI_VERSION 14
#define RZ_MAX_BOARD 19          /* rows live one per lane; A <= 362 (19x19 Go incl. the pass) */
#define RZ_META_STRIDE 12
#define RZ_GO_HIST 14            /* history planes a Go position carries besides the current board */

enum rz_meta {                   /* int32 words of a game's meta record */
  RZ_META_PLAYER = 0,            /* player to move, 0/1 (gomoku_env.py:29,67-68) */
  RZ_META_LAST_MOVE = 1,         /* -1 on an empty board (gomoku_env.py:45) */
  RZ_META_STONES = 2,            /* len(states) */
  RZ_META_STATUS = 3,            /* enum rz_status */
  RZ_META_WINNER = 4,            /* -1 none/tie, else player id (game_end_winner) */
  RZ_META_PLY = 5,               /* plies played in this episode (trajectory length) */
  RZ_META_FAULT = 6,             /* sticky bit set, enum rz_fault */
  RZ_META_EPISODE = 7,           /* episodes finished in this slot */
  RZ_META_KO = 8,                /* Go: square that may not be retaken, -1 none (go_base Position.ko) */
  RZ_META_PASSES = 9             /* Go: consecutive passes so far (two end the game, go_env.py:185) */
};                               /* words 10, 11 reserved.  Go also uses LAST_MOVE = last ACTION (the pass
                                    is H*W) and STONES = moves played (Position.n) */

enum rz_status {
  RZ_ACTIVE = 0,
  RZ_ENDED_WIN = 1,
  RZ_ENDED_TIE = 2,
  RZ_IDLE = 3                    /* waiting for the other seat (rz_match_commit): the game runs, but this forest's
                                    root is not the mover's; every tree kernel skips it like a finished game */
};

enum rz_fault {
  RZ_FAULT_ILLEGAL_MOVE = 1,     /* AssertionError in gomoku_env.py:51 */
  RZ_FAULT_POOL_OVERFLOW = 2,    /* node pool exhausted: leaf left unexpanded */
  RZ_FAULT_DEPTH_OVERFLOW = 4,
  RZ_FAULT_LN_TABLE = 8,         /* parent visit count beyond ln table */
  RZ_FAULT_NO_CHILDREN = 16,     /* ValueError in node.py:39 */
  RZ_FAULT_CARRY_DROPPED = 32,   /* reused subtree larger than max_carry: tree reset */
  RZ_FAULT_TRAJ_OVERFLOW = 64
};

enum rz_rule {
  RZ_RULE_UCT = 0,               /* reference: W/n + c*sqrt(ln(Np)/n), +inf if n==0 (node.py:75-88) */
  RZ_RULE_PUCT = 1               /* (n and W/n) + c*P*sqrt(Np)/(n+1) (deepmind_mcts.py:149-151) */
};

enum rz_flavour {                /* which of the reference's two search drivers the kernels follow */
  RZ_FLAVOUR_ALPHAZERO = 0,      /* AlphaZeroMCTS (rlzero/mcts/alphazero_mcts.py:42-103): scalar value, sign flip */
  RZ_FLAVOUR_DEEPMIND = 1        /* DeepMindMCTS (rlzero/mcts/deepmind_mcts.py:384-646, the OpenSpiel bot): returns
                                    vector indexed by the player who moved, outcome shortcut in the child score
                                    (:123-124,146-147), terminal outcomes, optional MCTS-Solver backup (:617-642),
                                    root-only Dirichlet noise (:484-485), search stops once the root is proven */
};

enum rz_returns {                /* env.returns() of a finished game, indexed by player */
  RZ_RETURNS_REFERENCE = 0,      /* bug-compatible with GomokuEnv.returns (gomoku_env.py:210-225): it tests winner
                                    == 1 / == 2 while players are 0 / 1, so a win of player 1 yields [1,-1] and
                                    everything else [0,0].  Go (go_env.py:142-143,350-354): [1,-1] if black won
                                    else [-1,1] -- already consistent */
  RZ_RETURNS_ZERO_SUM = 1        /* the evident intent: +1 for the winner, -1 for the loser, [0,0] for a tie */
};

enum rz_eval {                   /* closed-form evaluators, oracle/evaluators.py */
  RZ_EVAL_ZERO = 0, RZ_EVAL_KAT = 1, RZ_EVAL_HASH = 2
};

enum rz_child {                  /* values of edge child[] when N >= 1 */
  RZ_CHILD_TERMINAL = -1,        /* visited, game over there: never expanded (alphazero_mcts.py:60-68) */
  RZ_CHILD_OVERFLOW = -2,        /* visited, pool was full: re-evaluated like a leaf */
  RZ_CHILD_PENDING = -3          /* leaf-parallel mode only: a playout of the current wave is in flight through
                                    this never-visited edge (its visit count is virtual) */
};

/* ---- game geometry ------------------------------------------------------- */
enum rz_game {
  RZ_GAME_GOMOKU = 0,            /* k-in-a-row, action = square r*W+c (gomoku_env.py; TicTacToe = 3x3, k=3) */
  RZ_GAME_CONNECT4 = 1,          /* k-in-a-row with gravity: action = column, the stone drops to the lowest
                                    empty row (row 0 = bottom).  No reference env exists (SURVEY 0); same
                                    duck-typed API, planes and win rule as GomokuEnv */
  RZ_GAME_GO = 2                 /* Go as rlzero/games/go/go_env.py plays it through pettingzoo's go_base
                                    (MiniGo rules): captures, no suicide, simple ko, action H*W = pass, two
                                    passes end the game, Tromp-Taylor area score minus komi; player 0 = black */
};

typedef struct rz_game_desc {
  int32_t board_size;            /* H: rows      (GomokuEnv.board_size; H == W for Gomoku) */
  int32_t n_in_row;              /* k            (GomokuEnv.n_in_row) */
  int32_t n_actions;             /* A = H*W (Gomoku) or W (Connect Four) */
  int32_t action_stride;         /* AS = round_up(A, 32) */
  int32_t width;                 /* W: columns (0 means W = H) */
  int32_t game_type;             /* enum rz_game */
  float komi;                    /* Go: points given to white (GoEnv komi, go_env.py:41); 0 otherwise */
  int32_t max_moves;             /* Go: > 0 ends and scores the game after that many moves (engine-side cap,
                                    the reference has none); 0 = no cap */
  int32_t row_stride;            /* network kernels only: row stride S of the padded position layout the trunk
                                    activations use (a board owns S*S rows, square (y,x) at row y*S+x).
                                    0 = the smallest of 8 / 16 / 20 with max(H,W) < S; else exactly 8, 16 or 20 */
} rz_game_desc;

/* ---- one search forest: G trees, one per game ---------------------------- */
typedef struct rz_tree_desc {
  rz_game_desc game;
  int32_t n_trees;               /* G */
  int32_t max_nodes;             /* expanded-node capacity per tree */
  int32_t max_depth;             /* path capacity per tree (<= A+1) */
  int32_t rule;                  /* enum rz_rule */
  int32_t ln_table_len;
  int32_t store_priors;          /* 0: edge_P may be NULL (UCT ignores priors, SURVEY 0) */
  double c_puct;                 /* AlphaZeroMCTS._c_puct */
  int64_t global_offset;         /* global id of tree 0 (shard-invariant RNG streams) */
  /* node pools, [G][max_nodes][AS] */
  int32_t* edge_N;
  double* edge_W;
  float* edge_P;
  int32_t* edge_child;
  /* node headers, [G][max_nodes] */
  int32_t* node_parent;          /* -1 for the root */
  int32_t* node_paction;         /* action leading here from the parent */
  /* per tree, [G] */
  int32_t* n_nodes;              /* expanded nodes in use; 0 <=> root is an unexpanded leaf */
  int32_t* root_N;               /* TreeNode.explore_count of the root */
  double* root_W;                /* TreeNode.total_reward of the root */
  /* root positions */
  uint32_t* root_rows;           /* [G][2][H] */
  int32_t* root_meta;            /* [G][RZ_META_STRIDE] */
  /* per-wave scratch written by rz_tree_select, read by eval / expand_backup */
  int32_t* path_node;            /* [G][max_depth] */
  int32_t* path_action;          /* [G][max_depth] */
  int32_t* depth;                /* [G]; -1 = tree skipped this wave */
  uint32_t* leaf_rows;           /* [G][2][H] */
  int32_t* leaf_meta;            /* [G][RZ_META_STRIDE] (status = terminal state of the leaf) */
  const double* ln_table;        /* ln_table[k] = math.log(k) computed by the HOST libm (k>=1) */
  /* Go only (NULL otherwise): board_history planes 2..15 of go_env.py:174-178, [G][RZ_GO_HIST][H] */
  uint32_t* root_hist;
  uint32_t* leaf_hist;
  /* DeepMindMCTS flavour only (NULL / 0 otherwise) */
  int32_t flavour;               /* enum rz_flavour */
  int32_t solve;                 /* DeepMindMCTS(solve=...): back proven outcomes up the path */
  int32_t returns_mode;          /* enum rz_returns */
  int32_t noise_root_only;       /* Dirichlet noise only when the expanded node is the root (deepmind_mcts.py:484) */
  int32_t* edge_O;               /* [G][max_nodes][AS] SearchNode.outcome of each child: 0 = None, else
                                    0x100 | (outcome[0]+1) | (outcome[1]+1) << 2 */
  int32_t* root_O;               /* [G] outcome of the root, same encoding */
  /* leaf-parallel waves with virtual loss (opt-in, AlphaZero flavour; NOT the reference's sequential order --
     leaves_per_tree <= 1 is the parity mode and ignores the other three fields).  Every tree runs up to K
     playouts per wave: the warp that owns the tree descends K times in a row, and after each descent adds one
     virtual visit and subtracts virtual_loss from the value sum of every edge on that path (no atomics needed:
     one warp per tree), so the next descent is steered elsewhere.  rz_tree_expand_backup first restores the
     edges exactly (saved value sums, reverse order), then expands and backs up the K leaves in order; a leaf
     reached twice in one wave is expanded once and backed up twice.  All per-wave arrays (path_node,
     path_action, depth, leaf_rows, leaf_meta, leaf_hist, the evaluator's prior / value) then hold G*K entries,
     leaf slot = tree*K + k. */
  int32_t leaves_per_tree;       /* K */
  int32_t* target_N;             /* [G] or NULL: a tree takes no playout once root_N reaches target_N (so the last
                                    wave of a search may be partial); a tree whose root is unexpanded takes one */
  double* vl_saved_W;            /* [G*K][max_depth] scratch: the value sums the virtual losses overwrote */
  double virtual_loss;           /* subtracted per in-flight playout (1.0 = a lost game for the mover) */
  /* optional pools / inputs (ABI 8; every one may be NULL) */
  double* edge_P64;              /* [G][max_nodes][AS] the priors in float64.  TreeNode.prior is a Python float: with
                                    Dirichlet noise the reference forms 0.75 * p + 0.25 * noise in float64
                                    (node.py:66-69), which a float32 pool cannot hold.  When non-NULL the PUCT rule
                                    reads this pool instead of edge_P, expand writes both */
  const unsigned long long* seed_dev; /* [1] device scalar added to the `seed` argument of rz_tree_expand_backup* and
                                    rz_eval_rollout*: a captured CUDA graph holds `seed` by value, the host bumps this
                                    word between searches instead of re-capturing */
  int32_t* edge_R;               /* [G][max_nodes][AS] DeepMindMCTS flavour: position of each child in its parent's
                                    `children` list, which the reference shuffles (deepmind_mcts.py:508) -- `max()`
                                    returns the FIRST maximum, so the list order is the tie-break of the child
                                    selection (:513-517) and of best_child (:173-175).  NULL = unshuffled (ties go to
                                    the lowest action).  Expansion fills it with counter-based random keys
                                    (shuffle_mode 1) or with the slot index (shuffle_mode 0: the host overwrites a
                                    node's ranks with the permutation numpy's RandomState.shuffle drew, the seeded
                                    parity path of rlzero_b200.mcts.DeepMindMCTS) */
  int32_t shuffle_mode;
  int32_t reserved0;
} rz_tree_desc;

/* ---- trajectory store (GameControl.start_self_play, game.py:96-134) ------- */
typedef struct rz_traj_desc {
  int32_t max_plies;             /* staging capacity per game (<= A) */
  int32_t ring_capacity;         /* finished-ply records the ring holds */
  /* staging, per game per ply */
  uint32_t* stage_rows;          /* [G][max_plies][2][H] position BEFORE the move */
  int32_t* stage_info;           /* [G][max_plies][4]: mover, last_move, move played, stones */
  float* stage_pi;               /* [G][max_plies][AS] */
  /* ring of finished plies (z known) */
  uint32_t* ring_rows;           /* [cap][2][H] */
  int32_t* ring_info;            /* [cap][6]: mover, last_move, z (+1/-1/0), slot, episode, ply */
  float* ring_pi;                /* [cap][AS] */
  unsigned long long* ring_cursor; /* [1] records ever written (monotone) */
  unsigned long long* games_done;  /* [1] */
  unsigned long long* plies_done;  /* [1] */
} rz_traj_desc;

int rz_abi_version(void);
const char* rz_last_error(void);                 /* host string, thread-local */
int rz_sizeof_tree_desc(void);
int rz_sizeof_traj_desc(void);

/* ---- game dynamics: GomokuEnv (rlzero/games/gomoku/gomoku_env.py) -------- */
/* reset (gomoku_env.py:33-47): empty boards, player 0 to move, last_move -1.
   only_ended != 0: touch only games whose status is ENDED_* (continuous refill). */
int rz_gomoku_reset(const rz_game_desc* g, uint32_t* rows, int32_t* meta, int n_games,
                    int only_ended, void* stream);
/* step (gomoku_env.py:49-70): place stone, win check, flip player.  actions[i] < 0
   skips game i.  reward/win may be NULL.  Illegal move -> RZ_FAULT_ILLEGAL_MOVE. */
int rz_gomoku_step(const rz_game_desc* g, uint32_t* rows, int32_t* meta, const int32_t* actions,
                   int32_t* reward, int32_t* win, int n_games, void* stream);
/* leagel_actions (gomoku_env.py:72-73) as a byte mask [n][A]. */
int rz_gomoku_legal_mask(const rz_game_desc* g, const uint32_t* rows, uint8_t* mask,
                         int n_games, void* stream);
/* has_a_winner / game_end_winner (gomoku_env.py:116-170,196-203): end[i] 0/1, winner[i]. */
int rz_gomoku_winner(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta,
                     int32_t* end, int32_t* winner, int n_games, void* stream);
/* current_state (gomoku_env.py:95-114) as float32 [n][4][H][W]. */
int rz_gomoku_encode_f32(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta,
                         float* planes, int n_games, void* stream);
/* the same planes channels-last, float32 [n][HW][4] (input of the fp32 trunk). */
int rz_gomoku_encode_nhwc_f32(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta,
                              float* planes, int n_games, void* stream);

/* ---- game dynamics: GoEnv (rlzero/games/go/go_env.py over pettingzoo go_base = MiniGo rules) ----
   Positions: rows [n][2][H] (black, white), hist [n][RZ_GO_HIST][H] = board_history planes 2..15
   (go_env.py:174-178; planes 0,1 are the current stones of the last mover / of the player to move),
   meta as above (+ KO, PASSES).  hist may be NULL where noted (history not tracked). */
/* reset (go_env.py:212-230): empty boards, black to move, no ko, zero history. */
int rz_go_reset(const rz_game_desc* g, uint32_t* rows, uint32_t* hist, int32_t* meta, int n_games,
                int only_ended, void* stream);
/* step (go_env.py:168-210): Position.play_move (captures, ko; action H*W = pass), history shift,
   is_game_over -> status / winner (black iff result() == 1, go_env.py:142-143).  actions[i] < 0
   skips game i.  reward [n][2] (black, white) = GoEnv.rewards, done [n]; both may be NULL.
   Illegal move (occupied, ko, suicide, or the game is over) -> RZ_FAULT_ILLEGAL_MOVE.  hist may be NULL. */
int rz_go_step(const rz_game_desc* g, uint32_t* rows, uint32_t* hist, int32_t* meta, const int32_t* actions,
               int32_t* reward, int32_t* done, int n_games, void* stream);
/* Position.all_legal_moves (go_env.py:193-194) as a byte mask [n][H*W + 1] (only the pass once the
   game is over, go_env.py:192). */
int rz_go_legal_mask(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta, uint8_t* mask,
                     int n_games, void* stream);
/* Position.score() (Tromp-Taylor area, komi subtracted) as float64 [n] and result() in {1,-1,0} [n];
   either may be NULL. */
int rz_go_score(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta, double* score,
                int32_t* result, int n_games, void* stream);
/* observe (go_env.py:156-166) as float32 [n][17][H][W]: the 16 history planes + the player plane
   (channels first; the reference's array is [H][W][17]).  hist NULL = zero history. */
int rz_go_encode_f32(const rz_game_desc* g, const uint32_t* rows, const uint32_t* hist, const int32_t* meta,
                     float* planes, int n_games, void* stream);

/* ---- search: AlphaZeroMCTS (rlzero/mcts/alphazero_mcts.py, node.py) ------- */
/* fresh trees: _root = TreeNode(None, 1.0) (alphazero_mcts.py:36).  tree_mask NULL = all. */
int rz_tree_reset(const rz_tree_desc* t, const uint8_t* tree_mask, void* stream);
/* descent of one playout per tree (alphazero_mcts.py:48-54 + node.py:32-42,75-88 +
   gomoku_env.py:49-70), then game_end_winner on the leaf (alphazero_mcts.py:60).  With
   t->leaves_per_tree = K > 1: up to K descents per tree, each followed by its virtual loss
   (see rz_tree_desc); the wave arrays hold G*K slots. */
int rz_tree_select(const rz_tree_desc* t, void* stream);
/* expand (node.py:44-73) + terminal value rule (alphazero_mcts.py:60-68) + sign-flipping
   backup (node.py:135-144).  prior: [G][AS] float32; prior_is_log != 0 means it holds
   log-probabilities and exp() is applied (alphazero_agent.py:43).  value: [G] float32 (the
   network's output type); value64 != NULL overrides it with [G] float64 (a Python
   policy_value_fn returns a Python float, alphazero_mcts.py:59).
   noise_eps > 0 mixes Dirichlet(noise_alpha) noise into every expanded node
   (node.py:63-69, eps = 0.25, alpha = 0.3), counter-based RNG keyed by (seed, game, node).
   Leaf-parallel mode: prior [G*K][AS], value [G*K]; the virtual losses of the wave are taken off first. */
int rz_tree_expand_backup(const rz_tree_desc* t, const float* prior, int prior_is_log,
                          const float* value, const double* value64, float noise_eps, float noise_alpha,
                          unsigned long long seed, void* stream);
/* rz_tree_expand_backup of wave w and rz_tree_select of wave w + 1 in ONE launch (one leaf per tree and wave only): the same
   results as the two calls in sequence, one kernel boundary less per wave.  `value64` as in rz_tree_expand_backup
   (AlphaZero flavour) / rz_tree_expand_backup_dm (DeepMindMCTS flavour: the evaluator's returns [G][2]).
   Replaces the tail of one _playout and the head of the next (rlzero/mcts/alphazero_mcts.py:41-71). */
int rz_tree_expand_backup_select(const rz_tree_desc* t, const float* prior, int prior_is_log, const float* value,
                                 const double* value64, float noise_eps, float noise_alpha, unsigned long long seed,
                                 void* stream);
/* the same step with host-supplied randomness (seeded parity with the reference, whose noise comes from the global
   numpy stream, node.py:63-69; SURVEY 8 b2 `noise*|NULL`).  Either of
     noise64 [G*K][AS] float64: a Dirichlet sample per leaf, entry s = the noise of the child reached by action s
                                 (the reference indexes it by position in the legal-move list): the priors become
                                 (double)((1 - eps)_f32 * p_f32) + eps * noise64[s], numpy's arithmetic for a float32 p
                                 (eps = noise_eps; no device draw);
     prior64 [G*K][AS] float64: the finished float64 priors of the new node, stored verbatim (prior / noise_* ignored);
   both NULL = rz_tree_expand_backup.  With t->edge_P64 the float64 values are kept, else rounded to float32. */
int rz_tree_expand_backup_ex(const rz_tree_desc* t, const float* prior, int prior_is_log,
                             const float* value, const double* value64, float noise_eps, float noise_alpha,
                             unsigned long long seed, const double* noise64, const double* prior64, void* stream);
/* DeepMindMCTS flavour of the same step (deepmind_mcts.py:596-644): `value` is the evaluation for the
   player to move at the leaf (returns = [v,-v] in player order); ret64 != NULL overrides it with the
   evaluator's full returns vector, float64 [G][2] (Evaluator.evaluate, :22-24).  Terminal leaves take
   env.returns() per t->returns_mode and record it as the node's outcome; with t->solve the proven
   outcomes are backed up (MCTS-Solver). */
int rz_tree_expand_backup_dm(const rz_tree_desc* t, const float* prior, int prior_is_log, const float* value,
                             const double* ret64, float noise_eps, float noise_alpha, unsigned long long seed,
                             void* stream);
/* SearchNode.best_child (deepmind_mcts.py:153-175): argmax over the root's children of
   (outcome[player] or 0, explore_count, total_reward), first maximum; best[g] = -1 if the root has no
   children.  outcome_out (may be NULL) [G] = the root's outcome code (0 = unproven). */
int rz_tree_best_child(const rz_tree_desc* t, int32_t* best, int32_t* outcome_out, void* stream);
/* root statistics + move choice (alphazero_mcts.py:86-94, 144-148):
   visits int32 [G][AS] (0 where no child), pi float32 [G][AS] = softmax(log(N+1e-10)/T),
   move[g] sampled from pi with a counter-based RNG (seed, game, ply); u01 != NULL supplies
   the uniforms instead (tests).  Any output may be NULL. */
int rz_tree_root_policy(const rz_tree_desc* t, double temperature, int32_t* visits, float* pi,
                        int32_t* move, const double* u01, unsigned long long seed, void* stream);
/* play moves[g] on the root position and re-root (update_with_move, alphazero_mcts.py:96-103):
   keep_subtree != 0 compacts the chosen child's subtree to the front of the pool (self-play),
   else the tree is reset (play mode :157-158).  moves[g] < 0 resets the tree without a move
   (reset_player, :132-134).  traj != NULL records (position, pi, mover) first and, when the
   game ends, assigns z and flushes the episode to the ring (game.py:113-134); auto_reset != 0
   then restarts the slot from an empty board. */
int rz_tree_advance(const rz_tree_desc* t, const int32_t* moves, int keep_subtree, int max_carry,
                    const rz_traj_desc* traj, const float* pi, int auto_reset, void* stream);

/* ---- evaluation matches: GameControl.start_play (rlzero/games/gomoku/game.py:61-94) for G games at once ----
   Two forests, one per seat, over the same G games: tree g of each forest is game g.  In a running game exactly
   one seat's root is RZ_ACTIVE (the mover's), the other's RZ_IDLE.  For every game whose seat-s root is ACTIVE
   the move is moves_s[g] (rz_tree_root_policy's draw on that forest) or, when moves_s is NULL, the first
   most-visited child of the root (RolloutMCTS.simulate, rollout_mcts.py:76-81).  The move is played and logged
   at move_log[g * max_plies + ply]; both roots receive the new position and fresh trees; the mover's root turns
   IDLE and the other ACTIVE, or both take the ended status and the winner.  An illegal move raises
   RZ_FAULT_ILLEGAL_MOVE, an unexpanded mover root RZ_FAULT_NO_CHILDREN, in the mover's root meta (nothing is
   played then).  Line games, AlphaZero flavour, one leaf per wave; max_plies >= the board's cells. */
int rz_match_commit(const rz_tree_desc* seat0, const rz_tree_desc* seat1, const int32_t* moves0,
                    const int32_t* moves1, int32_t* move_log, int max_plies, void* stream);

/* ---- closed-form evaluators for parity tests (oracle/evaluators.py) ------- */
int rz_eval_closed_form(const rz_tree_desc* t, int eval_id, float* prior, float* value,
                        void* stream);

/* ---- training-side data path (tools/train_alphazero.py:59-90), SURVEY 8 f1 ----------------------
   get_equi_data: the 8 symmetric copies of n recorded plies, in the reference's order (for i in
   1..4: rot90^i, then its fliplr).  rows [n][2][H], info [n][info_stride] int32 (mover, last_move, z,
   ...: the trajectory ring's records), pi f32 [n][AS]  ->  out_planes f32 [8n][4][H][W] (current_state
   of the transformed position), out_pi f32 [8n][A], out_z f32 [8n].  Square Gomoku boards only: any other
   game_type or width is rejected on the host (Go records go through rz_go_records_pack / _expand). */
int rz_augment_equi(const rz_game_desc* g, const uint32_t* rows, const int32_t* info, int info_stride,
                    const float* pi, float* out_planes, float* out_pi, float* out_z, int n, void* stream);
/* Go training records (g: an RZ_GAME_GO descriptor, A = H*H + 1, AS = action_stride).  n trajectory-ring records in
   drain order -- rows [n][2][H], info [n][info_stride >= 6] int32 (mover, last_move, z, slot, episode, ply), pi f32
   [n][AS] -- are packed into a caller-owned ring of `capacity` compact records: planes uint32 [capacity][16][H] (the
   first 16 GoEnv.observe planes as row bitmasks: entry e = 0..7 is the position e plies back as (stones of its previous
   mover, stones of its mover), rebuilt from the preceding records of the same slot and episode, zero where there is
   none -- BatchedSelfPlay._go_states), mover int32 [capacity], pi f32 [capacity][A], z f32 [capacity].  Record i goes
   to slot (dst_start + i) % capacity; every input record serves as history, but with n > capacity only the newest
   capacity are written.  2672 bytes per position at 19x19. */
int rz_go_records_pack(const rz_game_desc* g, const uint32_t* rows, const int32_t* info, int info_stride,
                       const float* pi, int n, uint32_t* planes, int32_t* mover, float* out_pi, float* z, int capacity,
                       int dst_start, void* stream);
/* n (slot, symmetry) pairs of such a ring -> out_states f32 [n][17][H][H] (plane 16 = mover == 1, GoEnv.observe),
   out_pi f32 [n][A], out_z f32 [n]: what AlphaZeroAgent.learn takes.  Symmetry s: rot90 (s / 2 + 1) times, then fliplr
   when s is odd (rz_augment_equi's plane maps; s = 6 is the identity), applied to the planes AND to the H*H square
   probabilities; the pass is unchanged.  slots / syms are device int64; only slot % capacity and sym & 7 are read. */
int rz_go_records_expand(const rz_game_desc* g, const uint32_t* planes, const int32_t* mover, const float* pi,
                         const float* z, int capacity, const long long* slots, const long long* syms, int n,
                         float* out_states, float* out_pi, float* out_z, void* stream);
/* dst[i][:] = src[index[i]][:] for a [.][width] float table: mini-batch gather from the replay buffer
   (random.sample(self.data_buffer, batch_size), tools/train_alphazero.py:94). */
int rz_gather_rows(const float* src, const long long* index, float* dst, int n, int width, void* stream);

/* ---- the training step: AlphaZeroAgent.learn (rlzero/games/gomoku/alphazero_agent.py:59-86), SURVEY 8 f1 ----------
   Hand-written forward-with-saved-activations / analytic backward / loss / Adam in float32 (rz_learn.cu): no autograd,
   no cuDNN, no cuBLAS; every batch reduction in a fixed order (deterministic).  Activations are channels-last
   [n][HW][C] float32 (the layout of rz_net_conv3x3_f32, which is the forward convolution and -- with the weights
   rz_learn_pack_conv writes -- the data gradient); parameter gradients come out in the state_dict layouts.  The host
   mirror is rlzero_b200/learn.py::NativeTrainer; the oracle is oracle/train_oracle.py. */
/* C[M][N] = alpha * sum_k A(m,k) B(k,n) (+ C if accumulate); A(m,k) = A[m*sam + k*sak], B(k,n) = B[k*sbk + n*sbn]: every
   fully connected layer and its two gradients (nn.Linear, policy_value_net.py:20,24,25) */
int rz_learn_sgemm(int M, int N, int K, const float* A, long long sam, long long sak, const float* B, long long sbk,
                   long long sbn, float* C, long long ldc, float alpha, int accumulate, void* stream);
/* out[c] = alpha * sum_r in[r*ld + c] (bias gradients); scratch: n_slices * cols floats */
int rz_learn_colsum(const float* in, long long rows, int cols, long long ld, float* out, float alpha, float* scratch,
                    int n_slices, void* stream);
/* nn.Conv2d weight [cout][cin][3][3] -> w_fwd [tap][cin][cout] (rz_net_conv3x3_f32's layout) and w_bwd
   [8-tap][cout][cin]: rz_net_conv3x3_f32(dz, w_bwd, zero bias, ..., c_in = cout, c_out = cin) is the data gradient.
   Either output may be NULL. */
int rz_learn_pack_conv(const float* w_oihw, float* w_fwd, float* w_bwd, int c_in, int c_out, void* stream);
/* grad[i] = act[i] > 0 ? grad[i] : 0  (F.relu backward) */
int rz_learn_relu_bwd(const float* act, float* grad, long long n, void* stream);
/* [n][C][HW] -> [n][HW][C] */
int rz_learn_nchw_to_nhwc(const float* in, float* out, int n, int channels, int hw, void* stream);
/* dw [cout][cin][3][3] = sum over boards and squares of x (shifted by the tap) * dz, db [cout] = sum dz; x [n][HW][cin],
   dz [n][HW][cout]; c_in <= 64, c_out <= 128; scratch: 96 * 9 * c_in * c_out floats */
int rz_learn_conv_wgrad(const float* x, const float* dz, float* dw_oihw, float* db, float* scratch,
                        long long scratch_floats, int n_boards, int board_size, int c_in, int c_out, void* stream);
/* feat [n][6][HW] = relu(act_conv1 / val_conv1 (a3)) (policy_value_net.py:41,47); a3 [n][HW][128], w1x1 [6][128] */
int rz_learn_head_feat_fwd(const float* a3, const float* w1x1, const float* b1x1, float* feat, int n_boards, int hw,
                           void* stream);
/* logits[b][:] <- log_softmax(logits[b][:n_actions] + bias) in place, 0 in the padding (policy_value_net.py:43-44) */
int rz_learn_logsoftmax(float* logits, const float* bias, int n, int n_actions, int action_stride, void* stream);
/* h [n][64] <- relu(h + bv1) in place; v[b] = tanh(h[b] . wv2 + bv2) (policy_value_net.py:49-51) */
int rz_learn_value_fwd(float* h, const float* bv1, const float* wv2, const float* bv2, float* v, int n, void* stream);
/* loss and the gradients at the outputs (alphazero_agent.py:70-75,83-85): dlogits [n][AS] = (softmax * sum(pi) - pi) / n,
   dpre2 [n] = 2 (v - z) / n * (1 - v^2), dh [n][64] = dpre2 * wv2 * (h > 0); loss3 = (mse(v, z), -mean sum pi log p,
   -mean sum p log p).  terms: [n][3] scratch, scratch: 24 floats */
int rz_learn_loss_bwd(const float* logp, const float* pi, int pi_stride, const float* v, const float* z, const float* h,
                      const float* wv2, float* dlogits, float* dpre2, float* dh, float* terms, float* loss3,
                      float* scratch, int n, int n_actions, int action_stride, void* stream);
/* backward of the two 1x1 head convolutions: da3 [n][HW][128] = dfeat . w1x1, dw1x1 [6][128], db1x1 [6]; dfeat
   [n][6][HW] must already carry the ReLU mask; scratch: (ceil(n*HW/64) + 64) * 774 floats */
int rz_learn_head_feat_bwd(const float* dfeat, const float* a3, const float* w1x1, float* da3, float* dw1x1, float* db1x1,
                           float* scratch, long long scratch_floats, int n_boards, int hw, void* stream);
/* torch.optim.Adam on one flat buffer (L2 weight decay folded into the gradient, bias-corrected moments); step >= 1 */
int rz_learn_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, void* stream);

/* ---- the same step for the 128-channel ResNet trunk on the tensor cores (rz_learn_tc.cu) -------------------------
   bf16 activations / gradients in the padded position layout of the inference path, fp32 statistics and parameter
   gradients.  Row stride S = 16 up to 15x15 ([n*256][128]; forward convolution and data gradient through
   rz_net_conv3x3_tc2) or 20 up to 19x19 ([round_up(n*400, 256)][128]; rz_net_conv3x3_tc3); the data gradient runs
   with w_bwd below; the heads run through the float32 kernels above after rz_learn_tile_to_nhwc[_ex].  The _ex entry
   points take the row stride (16 or 20, anything else is an error naming row_stride); each plain entry point is the
   S = 16 call of its _ex form.  Tensors of stride S have round_up(n*S*S, 256) rows; a row is off the board when its
   x >= W, its y >= H, or the row is >= n*S*S, and off-board rows are written as zero. */
/* dw [128][128][3][3] fp32 = sum over positions of dy[p][co] * x[p + d(tap)][ci]: tcgen05 GEMM with MN-major operands
   (the reduction index is the tile row), accumulators in TMEM for the whole launch, CTA triples (one per filter row)
   sharing position tiles through L2.  x, dy: bf16 [n*256][128] with zero pad squares.  scratch: 49 * 9 * 128 * 128
   floats (per-split partials, folded in a fixed order).  n_ctas <= 0 picks 147. */
int rz_learn_conv_wgrad_tc(const void* x, const void* dy, float* dw_oihw, float* scratch, long long scratch_floats,
                           int n_boards, int n_ctas, void* stream);
/* the same at row stride S (16 or 20): x tiles carry an (S + 1)-row halo, ceil(n*S*S / 128) position tiles, which at
   S = 20 straddle boards (harmless: pad squares are zero); x, dy bf16 [round_up(n*S*S, 256)][128] */
int rz_learn_conv_wgrad_tc_ex(const void* x, const void* dy, float* dw_oihw, float* scratch, long long scratch_floats,
                              int n_boards, int row_stride, int n_ctas, void* stream);
/* nn.Conv2d weight fp32 [128][128][3][3] -> bf16 w_fwd [tap][cout][cin] (rz_net_conv3x3_tc2's layout) and w_bwd
   [8-tap][cin][cout]: rz_net_conv3x3_tc2(dy, w_bwd, zero bias, residual = skip gradient, ...) is the data gradient */
int rz_learn_pack_conv_tc(const float* w_oihw, void* w_fwd, void* w_bwd, void* stream);
/* inference weights of a 128 -> 128 trunk layer from the float32 parameters on the device: nn.Conv2d weight
   [128][128][3][3] (+ bias) with an eval-mode nn.BatchNorm2d folded in (gamma NULL = no BatchNorm; float64 arithmetic)
   -> bf16 [tap][cout][cin] and fp32 bias [128], the operands of rz_net_conv3x3_tc2 / _tc3: re-packing after a training
   step is one launch per layer, no host round trip */
int rz_net_pack_conv_bn_tc(const float* w_oihw, const float* conv_bias, const float* gamma, const float* beta,
                           const float* running_mean, const float* running_var, float eps, void* w_out, float* b_out,
                           void* stream);
/* stem weight fp32 [128][4][3][3] -> bf16 [128][64] (k = tap*4 + plane, rz_net_stem_tc's layout) */
int rz_learn_pack_stem_tc(const float* w_oihw, void* w_stem, void* stream);
/* in_planes 4: the same; in_planes 17 (Go): fp32 [128][17][3][3] -> bf16 [128][192] (k = tap*17 + plane, zero from 153:
   rz_net_stem_go_tc's layout) */
int rz_learn_pack_stem_tc_ex(const float* w_oihw, int in_planes, void* w_stem, void* stream);
/* nn.BatchNorm2d in training mode + skip + ReLU: batch statistics of y over the board squares (biased variance),
   running_mean / running_var updated (momentum, unbiased variance; may be NULL), out = relu((y - mean) * invstd *
   gamma + beta (+ skip)), zero off the board.  stats [4][128] receives mean, invstd, gamma * invstd, beta - mean *
   gamma * invstd (kept for the backward pass).  scratch: 148 * 4 * 256 + 256 floats. */
int rz_learn_bn_forward(const void* y, const void* skip, void* out, const float* gamma, const float* beta,
                        float* running_mean, float* running_var, float eps, float momentum, float* stats, float* scratch,
                        int n_boards, int board_rows, int board_cols, void* stream);
/* its backward pass: dz = dout * (act > 0); dgamma = sum dz * xhat, dbeta = sum dz; dy = gamma * invstd * (dz - dbeta / N -
   xhat * dgamma / N) (bf16, zero off the board); dz_out (may be NULL) receives dz, the gradient into the skip */
int rz_learn_bn_backward(const void* dout, const void* act, const void* y, const float* stats, float* dgamma, float* dbeta,
                         void* dy, void* dz_out, float* scratch, int n_boards, int board_rows, int board_cols, void* stream);
/* both at row stride S (boards up to S - 1 squares a side; the statistics still count n * H * W squares) */
int rz_learn_bn_forward_ex(const void* y, const void* skip, void* out, const float* gamma, const float* beta,
                           float* running_mean, float* running_var, float eps, float momentum, float* stats, float* scratch,
                           int n_boards, int board_rows, int board_cols, int row_stride, void* stream);
int rz_learn_bn_backward_ex(const void* dout, const void* act, const void* y, const float* stats, float* dgamma,
                            float* dbeta, void* dy, void* dz_out, float* scratch, int n_boards, int board_rows,
                            int board_cols, int row_stride, void* stream);
/* float32 observation planes [n][4][H][W] -> bf16 tile [n*256][128] (channels 0..3, rest zero): the stem's input as the
   x operand of rz_learn_conv_wgrad_tc (its result's input channels 0..3 are the stem's weight gradient) */
int rz_learn_planes_to_tile(const float* planes, void* tile, int n_boards, int board_rows, int board_cols, void* stream);
/* float32 planes [n][n_planes][H][W] (n_planes 4 or 17) -> bf16 tile of stride S, channels 0..n_planes-1 */
int rz_learn_planes_to_tile_ex(const float* planes, int n_planes, void* tile, int n_boards, int board_rows, int board_cols,
                               int row_stride, void* stream);
/* float32 channels-last [n][HW][C] -> bf16 tiles holding the values as (high, low) pairs (hi = bf16(x), lo = bf16(x - hi)):
   mode 0: tile_a[:, 0:C] = hi, tile_a[:, C:2C] = lo (2C <= 128; the layer input); mode 1: tile_a[:, 0:C] = hi,
   tile_b[:, 0:C] = lo (the output gradient).  Two rz_learn_conv_wgrad_tc launches (x pair-tile against the high and the
   low gradient tile) then hold all four partial products of the float32 weight gradient. */
int rz_learn_nhwc_to_tile_hilo(const float* in, int channels, void* tile_a, void* tile_b, int mode, int n_boards,
                               int board_rows, int board_cols, void* stream);
/* the same for a slice [channel_offset, channel_offset + channels) of a wider tensor (mode 0 layout, 2*channels <= 128) */
int rz_learn_nhwc_to_tile_hilo_slice(const float* in, int channels_total, int channel_offset, int channels, void* tile_a,
                                     int n_boards, int board_rows, int board_cols, void* stream);
/* float32 tile [n*256][128] (first `channels` channels) -> float32 channels-last [n][HW][channels] */
int rz_learn_tile_f32_to_nhwc(const float* tile, float* out, int channels, int n_boards, int board_rows, int board_cols,
                              void* stream);
/* data gradient of a float32-accurate layer in tile space: g = (grad_a + grad_b) * (act > 0) on the first `channels`
   channels (grad_a / grad_b: float32 tiles written by rz_net_conv3x3_tc2 with flag 64, grad_b may be NULL; act_pair: the
   layer's activation as a bf16 [hi | lo] pair tile).  g overwrites grad_a (float32) and leaves as bf16 pairs: pair_out =
   [hi | lo] in one tile (may be NULL), hi_out / lo_out separately (the gradient operands of rz_learn_conv_wgrad_tc) */
int rz_learn_tile_grad_mask_split(float* grad_a, const float* grad_b, const void* act_pair, int channels, void* pair_out,
                                  void* hi_out, void* lo_out, int n_boards, void* stream);
/* out[c] = sum over the rows of a bf16 tile [n*256][128] (a bias gradient); scratch: 148 * 2 * 256 floats */
int rz_learn_tile_colsum(const void* tile, float* out, float* scratch, int n_boards, void* stream);
int rz_learn_tile_colsum_ex(const void* tile, float* out, float* scratch, int n_boards, int row_stride, void* stream);
/* grad = dout * (act > 0) on bf16 tiles (ReLU without BatchNorm: the stem) */
int rz_learn_relu_bwd_bf16(const void* dout, const void* act, void* grad, int n_boards, void* stream);
int rz_learn_relu_bwd_bf16_ex(const void* dout, const void* act, void* grad, int n_boards, int row_stride, void* stream);
/* bf16 padded tile layout [n*256][128] <-> float32 [n][HW][128] */
int rz_learn_tile_to_nhwc(const void* tile, float* out, int n_boards, int board_rows, int board_cols, void* stream);
int rz_learn_nhwc_to_tile(const float* in, void* tile, int n_boards, int board_rows, int board_cols, void* stream);
int rz_learn_tile_to_nhwc_ex(const void* tile, float* out, int n_boards, int board_rows, int board_cols, int row_stride,
                             void* stream);
int rz_learn_nhwc_to_tile_ex(const float* in, void* tile, int n_boards, int board_rows, int board_cols, int row_stride,
                             void* stream);

/* ---- pure-MCTS opponent: random playouts (rlzero/mcts/rollout_mcts.py:49-74,96-108) ---------
   prior: uniform over the leaf's legal moves; value: the reference's _evaluate on a uniformly random
   playout from the leaf (at most n_limit plies; literal winner == current_player() rule, i.e. -1 for
   a decisive playout, 0 for a tie).  mode 0: counter-based RNG keyed by (seed, global game id, root
   visit count, ply); mode 1 / 2: always the lowest / highest legal move (deterministic tests). */
int rz_eval_rollout(const rz_tree_desc* t, int mode, unsigned long long seed, int n_limit, float* prior,
                    float* value, void* stream);

/* RandomRolloutEvaluator of the DeepMindMCTS driver (rlzero/mcts/deepmind_mcts.py:31-62): uniform priors
   over the leaf's legal actions and ret64 [G][2] = mean env.returns() (per t->returns_mode) of n_rollouts
   uniformly random playouts from the leaf (each at most n_limit plies; Go playouts include the pass and
   end by two passes or the move cap).  Feed ret64 to rz_tree_expand_backup_dm. */
int rz_eval_rollout_dm(const rz_tree_desc* t, int n_rollouts, unsigned long long seed, int n_limit,
                       float* prior, double* ret64, void* stream);

/* ---- policy-value network forward (rlzero/games/gomoku/policy_value_net.py:34-52) -------- */
/* heads weights, all float32 device pointers.  FC weights are stored TRANSPOSED ([in][out]);
   the flatten order of the FC inputs is c*HW + pos (x.view(-1, C*H*W) on NCHW, :42,48). */
typedef struct rz_heads_desc {
  int32_t board_size;            /* H rows */
  int32_t action_stride;         /* AS: row stride of wp / logp */
  int32_t width;                 /* W columns (0: W = H) */
  int32_t n_actions;             /* policy outputs (0: H*W) */
  int32_t row_stride;            /* S of the padded layout the features / trunk output use (0: automatic, as in
                                    rz_game_desc.row_stride) */
  const float* w1x1;             /* [6][128]  act_conv1 (4 filters) then val_conv1 (2 filters) */
  const float* b1x1;             /* [6] */
  const float* wp;               /* [4*HW + 4][AS] act_fc1.weight^T, zero padded (columns >= HW and the 4 extra rows) */
  const float* bp;               /* [AS] */
  const float* wv1;              /* [2*HW + 2][64] val_fc1.weight^T + 2 zero rows */
  const float* bv1;              /* [64] */
  const float* wv2;              /* [64]       val_fc2.weight */
  const float* bv2;              /* [1] */
  /* rz_net_heads_tc only (may be NULL otherwise): both FC weight matrices as ONE bf16 K-major matrix
     [AS + 64][KP], KP = round_up(6*S*S, 64), split into a high and a low part (w = hi + lo, lo = the bf16
     rounding error of hi).  Row a < AS: act_fc1.weight[a] at column f*S*S + y*S + x (f < 4; zero at padding
     squares and for a >= A); row AS + o: val_fc1.weight[o] at column (4 + f)*S*S + y*S + x (f < 2). */
  const void* wtc_hi;
  const void* wtc_lo;
} rz_heads_desc;

/* 3x3 convolution (padding 1) + bias (+ residual) (+ ReLU) on the tensor cores (tcgen05/TMEM/TMA), revision 2:
   nn.Conv2d + folded BatchNorm + ReLU of the trunk.
   act_in bf16 [n][256][c_in] in the padded tile layout described at the top of rz_net_tc2.cu (position
   p = y*16+x, zero pad squares), c_in in {64,128}; weight bf16 [9][128][c_in] (tap = kh*3+kw, then out channel,
   then in channel); bias f32 [128]; residual/act_out bf16 [n][256][128] (residual may alias act_out, may be NULL).
   The 9x128x128 weights stay resident in shared memory, split over a CTA pair (tcgen05 cta_group::2 MMAs, cluster
   of 2; cta_group must be 2), and each 128-position activation tile is loaded once with its 17-row halo; the 9 taps
   are row-shifted UMMA descriptors on that tile.  flags bit 0: set the base-offset field of the shifted
   descriptors; bit 1 (2) is accepted and ignored.  n_ctas <= 0 picks 148.
   Programmatic dependent launch: this kernel, rev. 3, the stems, the heads and the tree kernels of a wave are launched
   with cudaLaunchAttributeProgrammaticStreamSerialization and call griddepcontrol.wait before they read or write
   anything another kernel of the stream touches (RZ_PDL=0 in the environment turns it off).  flags bit 9 (512; for
   rev. 3: bit 1 of `relu`) = STATIC WEIGHTS: weight and bias are fetched BEFORE that wait, under the tail of the
   previous kernel -- the caller guarantees that the kernel launched immediately before on the stream does not
   write them (the search's forward pass: weights are packed at refresh_weights, which synchronises). */
int rz_net_conv3x3_tc2(const void* act_in, const void* weight, const float* bias, const void* residual,
                       void* act_out, int n_boards, int board_size, int board_cols, int c_in, int relu,
                       int cta_group, int flags, int n_ctas, void* stream);
/* the last trunk layer with the heads' two 1x1 convolutions + ReLU (act_conv1 128->4, val_conv1 128->2,
   policy_value_net.py:41,47) applied in its epilogue: writes ONLY feat f32 [n][6][256] (filter, then
   position p = y*16+x); the trunk output never reaches HBM.  w1x1_host [6][128] / b1x1_host [6] are
   HOST float32 arrays (copied into the launch parameters).  Feed feat to rz_net_heads_tc.
   flags 0, 512 (static weights, as above) or the kernel's mode flags: 16 = split input (act_in = [hi 0..63 | lo 0..63], the bf16 high parts and
   rounding residues of a 64-channel float32-accurate activation; weight = [tap][128][Whi 0..63 | Wlo 0..63]; three
   products per tap: hi*Whi + lo*Whi + hi*Wlo), 32 = the 1x1 head convolutions read the float32 accumulators instead
   of bf16-rounded activations.  Together: conv3 (64 -> 128) + act_conv1 / val_conv1 of the reference's own
   PolicyValueNet at float32-level accuracy on the tensor cores.  Likewise rz_net_conv3x3_tc2 accepts flags 8 =
   split output (64 real output channels written as [hi 0..63 | lo 0..63]), 64 = float32 output (act_out
   is float [rows][128]; no residual), 128 = only the first 96 input channels are issued, 256 = N = 64 MMAs
   for a layer with 64 output channels (with flag 8; weight rows 0..31 / 64..95 hold output channels 0..31 / 32..63), and
   the `relu` argument of
   rz_net_stem_tc / rz_net_stem_tc_planes bit 1 = 32-channel float32-accurate stem: weight rows 0..31 / 32..63 hold
   the high parts / residues of the 32 filters, the output row is [hi 0..31 | lo 0..31 | hi 0..31 | lo 0..31]. */
int rz_net_conv3x3_tc2_head_ex(const void* act_in, const void* weight, const float* bias, const void* residual,
                               int n_boards, int board_size, int board_cols, int c_in, int relu, int flags,
                               const float* w1x1_host, const float* b1x1_host, float* feat, int n_ctas,
                               void* stream);
/* small-batch latency path: the WHOLE 128-channel trunk of a board in one launch (the single-position evaluation of a
   sequential search, rlzero/mcts/alphazero_mcts.py:73-94).  One CTA pair per board keeps the activation in shared
   memory across all layers (ping-pong halo tiles written by the epilogue, the rows next to the seam between the two
   CTAs also into the peer's tile through distributed shared memory); the weights of all layers stream through a ring
   of taps; the MMAs, their order and the epilogue arithmetic are those of rz_net_conv3x3_tc2, so the results are
   bit-identical to n_layers launches of it followed by the fused-heads epilogue of rz_net_conv3x3_tc2_head_ex.
   act_in bf16 [n][256][128] (the stem's output); weights bf16 [n_layers][9][128][128] (layer, tap, out channel, in
   channel); biases f32 [n_layers][128]; bit l of relu_mask: ReLU after layer l; bit l of res_mask: layer l adds the
   input of layer l-1 (the block's skip connection) before its ReLU; feat f32 [n][6][256] as _tc2_head_ex.  n_layers <= 24.
   Weights and biases are STATIC in the sense of flag 512 above. */
int rz_net_trunk_small(const void* act_in, const void* weights, const float* biases, int n_layers,
                       unsigned relu_mask, unsigned res_mask, int n_boards, int board_size, int board_cols,
                       const float* w1x1_host, const float* b1x1_host, float* feat, void* stream);
/* the same with the modes of the float32-accurate path of the reference's own PolicyValueNet (flags 8 | 256 / 16 / 32 of
   rz_net_conv3x3_tc2[_head_ex]): bit l of n64_mask = layer l has 64 real output channels (N = 64 MMAs) and leaves as
   [hi 0..63 | lo 0..63]; bit l of split_in_mask = layer l takes such a row against weights [Whi | Wlo] (three products
   per tap); head_f32 = the 1x1 head convolutions read the float32 activations.  conv2 + conv3 + act_conv1 / val_conv1
   (policy_value_net.py:37-38,41,47) of one position in one launch, bit-identical to the two per-layer launches. */
int rz_net_trunk_small_ex(const void* act_in, const void* weights, const float* biases, int n_layers,
                          unsigned relu_mask, unsigned res_mask, unsigned n64_mask, unsigned split_in_mask, int head_f32,
                          int n_boards, int board_size, int board_cols, const float* w1x1_host,
                          const float* b1x1_host, float* feat, void* stream);
/* the same trunk for many boards (rz_net_trunk_tc2.cu): one launch on n_ctas / 2 CTA pairs (0 = 148 CTAs), pair p
   carrying a contiguous range of boards in chunks of at most `chunk` (1..16) boards through every layer, the activations
   between layers in `scratch` instead of act_in-sized tensors: bf16 [2][n_ctas / 2][chunk][256][128] (1 MB per pair at
   chunk 8; it must start zeroed, and the kernel keeps its pad rows zero).  act_in, weights, relu_mask, res_mask and
   feat as rz_net_trunk_small; biases_host f32 [n_layers][128] in host memory, copied into the launch parameters like
   w1x1_host.  Per board the MMAs and the epilogue arithmetic are those of rz_net_conv3x3_tc2[_head_ex], so the results
   are bit-identical to the per-layer launches and to rz_net_trunk_small.  Weights are STATIC as in flag 512 above. */
int rz_net_trunk_tc2(const void* act_in, const void* weights, const float* biases_host, int n_layers,
                     unsigned relu_mask, unsigned res_mask, void* scratch, int chunk, int n_boards, int board_size,
                     int board_cols, const float* w1x1_host, const float* b1x1_host, float* feat, int n_ctas,
                     void* stream);
/* profiling aid: rz_net_trunk_small writes four %globaltimer stamps per layer of board 0 (inputs ready / MMAs issued /
   accumulator complete / layer stored) into this device buffer of 4 * n_layers uint64; NULL (the default) = off. */
int rz_debug_set_probe(void* device_buffer);
/* revision 3 of the convolution: the same data path for any row stride of the padded position
   layout (row = board*S*S + y*S + x; S = row_stride = 8 for boards up to 7x7 such as Connect Four 6x7, 16 up
   to 15x15, 20 up to 19x19), tiles of 128 rows that may straddle boards (S = 20) or hold two boards (S = 8), a ring of k-block halo tiles (3 slots at S = 20, 4 at S = 8 / 16: the
   shared-memory budget of the 170-row halo) and rev. 2's direct-store epilogue.  c_in = c_out = 128.  Tensors are
   bf16 [round_up(n_boards*S*S, 256)][128].  The _head variant writes feat f32 [n_boards][6][S*S]. */
int rz_net_conv3x3_tc3(const void* act_in, const void* weight, const float* bias, const void* residual,
                       void* act_out, int n_boards, int board_rows, int board_cols, int row_stride, int relu,
                       int n_ctas, void* stream);
int rz_net_conv3x3_tc3_head(const void* act_in, const void* weight, const float* bias, const void* residual,
                            int n_boards, int board_rows, int board_cols, int row_stride, int relu,
                            const float* w1x1_host, const float* b1x1_host, float* feat, int n_ctas,
                            void* stream);
/* fused current_state (gomoku_env.py:95-114) + first trunk convolution (policy_value_net.py:14,36):
   the 36-wide im2col row of every position (k = tap*4 + plane) is built from the bitboards in
   registers, so the observation planes never exist in HBM.  weight bf16 [128][64] (k padded with
   zeros from 36), bias f32 [128], act_out bf16 [round_up(n*S*S, 256)][128] padded layout, S =
   g->row_stride, or when that is 0 the smallest of 8 (boards up to 7x7), 16 (up to 15x15, then
   [n][256][128]) and 20 (up to 19x19). */
int rz_net_stem_tc(const rz_game_desc* g, const uint32_t* rows, const int32_t* meta, const void* weight,
                   const float* bias, void* act_out, int n_boards, int relu, int n_ctas, void* stream);
/* the same kernel fed from float32 observation planes [n][4][H][W] (the current_state format,
   AlphaZeroAgent.policy_value / predict, alphazero_agent.py:48-57,88-97); planes are rounded to bf16. */
int rz_net_stem_tc_planes(const rz_game_desc* g, const float* planes, const void* weight, const float* bias,
                          void* act_out, int n_boards, int relu, int n_ctas, void* stream);
/* Go: fused GoEnv.observe (go_env.py:156-178: 16 history planes + player plane) + stem conv3x3(17->128):
   the 153-wide im2col row (k = tap*17 + plane) is built from the row bitmasks in registers.  weight bf16
   [128][192] (k zero padded from 153), bias f32 [128], act_out as rz_net_stem_tc (S = 16 up to 15x15, else 20).
   rows/hist/meta: the Go position records (rz_go_step).  The _planes variant reads float32 [n][17][H][W]. */
int rz_net_stem_go_tc(const rz_game_desc* g, const uint32_t* rows, const uint32_t* hist, const int32_t* meta,
                      const void* weight, const float* bias, void* act_out, int n_boards, int relu, int n_ctas,
                      void* stream);
int rz_net_stem_go_tc_planes(const rz_game_desc* g, const float* planes, const void* weight, const float* bias,
                             void* act_out, int n_boards, int relu, int n_ctas, void* stream);
/* the same operator in float32 on CUDA cores for the reference's stock network at any board size:
   in [n][HW][c_in], weight [9][c_in][c_out], out [n][HW][c_out] (channels last). */
int rz_net_conv3x3_f32(const float* in, const float* weight, const float* bias, const float* residual,
                       float* out, int n_boards, int board_size, int c_in, int c_out, int relu,
                       void* stream);
/* both heads on CUDA cores from the fp32 trunk output act f32 [n][HW][128] (channels last, as
   rz_net_conv3x3_f32 writes it): logp f32 [n][AS] = log_softmax(policy logits) (0 in the padding),
   value f32 [n] = tanh(...). */
int rz_net_heads(const rz_heads_desc* h, const float* act, float* logp, float* value, int n_boards, void* stream);
/* the heads' two 1x1 convolutions + ReLU alone (policy_value_net.py:41,47): act bf16 padded layout
   [n*S*S][128] -> feat f32 [n][6][S*S], the tensor rz_net_conv3x3_tc2_head_ex / _tc3_head write from their
   epilogue (same summation order: bit-identical at the board's squares). */
int rz_net_head_features(const rz_heads_desc* h, const void* act, float* feat, int n_boards, void* stream);
/* the fully connected layers of both heads on the tensor cores (act_fc1 + log_softmax, val_fc1 + ReLU +
   val_fc2 + tanh; policy_value_net.py:42-44,48-51) from feat f32 [n][6][S*S]: one tcgen05 GEMM per 128 boards
   over the padded feature row, bf16 hi/lo split of features and weights (3 MMAs per k-step) for float32-level
   accuracy, accumulators and the softmax in TMEM.  Needs h->wtc_hi / wtc_lo; logp f32 [n][AS], value f32 [n]. */
int rz_net_heads_tc(const rz_heads_desc* h, const float* feat, float* logp, float* value, int n_boards,
                    void* stream);

/* ---- MuZero search in latent space (BASELINE.json config 5) ----------------------------------------
   The reference has no MuZero code: the kernels follow the pseudocode published with the MuZero paper
   (run_mcts, select_child, ucb_score, expand_node, backpropagate, add_exploration_noise, MinMaxStats) with
   the two-player value-sign convention; rewards are 0 (board games).  PARITY UNPINNED (oracle/muzero_oracle.py).
   A node's children live in its edge block as in rz_tree_desc; W is the child's value_sum from the child's own
   to_play view.  Every simulation expands exactly one node, so node i+1 of every tree is created by simulation
   i and hidden states are stored node-major: pool[node][tree][S*S][128] bf16. */
typedef struct rz_mz_desc {
  int32_t n_trees;               /* G */
  int32_t n_actions;             /* A: the action space below the root */
  int32_t action_stride;         /* AS = round_up(A, 32) */
  int32_t max_nodes;             /* num_simulations + 1 */
  int32_t max_depth;             /* path capacity (<= max_nodes) */
  int32_t pbc_table_len;
  double discount;               /* MuZeroConfig.discount (1 for board games) */
  double known_min, known_max;   /* MinMaxStats known_bounds; +inf / -inf when unknown */
  int64_t global_offset;         /* global id of tree 0 (shard-invariant noise) */
  int32_t* edge_N;               /* [G][max_nodes][AS] visit_count of each child, -1 = no such child */
  double* edge_W;                /* value_sum */
  float* edge_P;                 /* prior */
  int32_t* edge_child;           /* node index once expanded, else -1 */
  int32_t* n_nodes;              /* [G] */
  int32_t* root_N;               /* [G] */
  double* root_W;                /* [G] */
  double* mm_min;                /* [G] MinMaxStats.minimum */
  double* mm_max;                /* [G] MinMaxStats.maximum */
  int32_t* path_node;            /* [G][max_depth] scratch of one simulation */
  int32_t* path_action;          /* [G][max_depth] */
  int32_t* depth;                /* [G] length of the search path below the root; -1 = fault */
  int32_t* leaf_parent;          /* [G] node whose hidden state feeds recurrent_inference */
  int32_t* leaf_action;          /* [G] history.last_action() */
  int32_t* fault;                /* [G] sticky bits: 1 = path/pb_c table overflow, 2 = node pool full */
  const double* pbc_table;       /* pbc_table[n] = log((n + pb_c_base + 1) / pb_c_base) + pb_c_init, HOST libm */
} rz_mz_desc;

int rz_sizeof_mz_desc(void);
/* expand_node(root, to_play, legal_actions, initial_inference) + add_exploration_noise: priors =
   exp(logp) renormalised over the legal actions (legal uint8 [G][A], NULL = all), mixed with
   Dirichlet(noise_alpha) noise when noise_eps > 0 (counter-based RNG keyed by seed, global tree id and the
   move counter: move_ids[g] when move_ids != NULL -- a device array, so a captured graph sees fresh counters --
   else move_id); fresh tree of one node, MinMaxStats reset to the known bounds. */
int rz_mz_root(const rz_mz_desc* t, const float* logp, const uint8_t* legal, float noise_eps, float noise_alpha,
               unsigned long long seed, unsigned int move_id, const int32_t* move_ids, void* stream);
/* the descent of one simulation (select_child until a child that is not expanded): fills path_*, depth,
   leaf_parent, leaf_action.  ucb_score in float64: pb_c = pbc_table[N] * (sqrt(N) / (n + 1)); score =
   pb_c * prior + (n > 0 ? normalize(discount * -value_sum / n) : 0); ties go to the HIGHEST action
   (max over (score, action) tuples). */
int rz_mz_select(const rz_mz_desc* t, void* stream);
/* expand_node(leaf, recurrent_inference) + backpropagate: new node n_nodes with priors exp(logp) over the
   whole action space (logp f32 [G][AS] = log_softmax of the prediction network), value f32 [G] for the
   player to move at the leaf. */
int rz_mz_expand_backup(const rz_mz_desc* t, const float* logp, const float* value, void* stream);
/* input of the dynamics network: stage[g] = pool[parent[g]][g] with channel 127 replaced by the one-hot
   plane of action[g] (an action >= rows*cols, Go's pass, gives an empty plane).  pool bf16
   [slots][slot_rows][128] with slot_rows >= n_trees*S*S, stage bf16 [n_trees*S*S][128], S = row_stride. */
int rz_mz_gather(const void* pool, const int32_t* parent, const int32_t* action, void* stage, int n_trees,
                 int board_rows, int board_cols, int row_stride, long long slot_rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RLZERO_B200_H */
