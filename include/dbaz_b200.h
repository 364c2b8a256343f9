/*
 * dbaz_b200.h -- C ABI of the B200-native Dots & Boxes AlphaZero self-play engine.
 *
 * The reference (damlobster/DotsBoxesAZ) is pure Python and has no FFI of its
 * own; its "operator API" for the self-play hot path is the Python surface of
 * game.py / dots_boxes/dots_boxes_game.py / mcts.py.  Each entry point below
 * names the reference function(s) it replaces (paths relative to the reference
 * root).  The Python binding a maintainer would add is in INTEGRATION.md and is
 * what dotsboxesaz_b200/_capi.py implements.
 *
 * Conventions
 *  - Every bulk buffer is a CALLER-OWNED DEVICE pointer (tensor.data_ptr()) of
 *    the stated element type and shape, C-contiguous; sizes are explicit.
 *  - `stream` is a cudaStream_t passed as an integer handle
 *    (torch.cuda.current_stream().cuda_stream); all work is enqueued on it, no
 *    entry point synchronises the device unless its comment says so.
 *  - Return value: 0 = OK, non-zero = error; dbaz_last_error() gives the text.
 *    Device-side faults (illegal move, node pool exhausted) are recorded per
 *    game and surfaced by dbaz_search_status(); nothing throws across the ABI.
 *  - A handle is not thread-safe; use one handle per GPU per process.
 *  - No CPU fallback exists: without a CUDA device dbaz_engine_create() fails.
 */
#ifndef DBAZ_B200_H
#define DBAZ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBAZ_ABI_VERSION 1
#define DBAZ_MAX_ACTIONS 128 /* A = 2*(L+1)*(C+1) <= 128, i.e. boards up to 7x7 boxes */
#define DBAZ_RESULT_NONE 2   /* get_result() is None */
#define DBAZ_MAX_PENDING 128 /* upper bound of max_pending_evals per tree */

/* Bit-packed game state, 32 bytes (dots_boxes_game.py:13, __slots__ hash/board/
 * just_played/to_play/boxes_to_close).  Bit a of `edges` is set iff
 * board.ravel()[a] == 255; padding cells are implied by the board size. */
typedef struct dbaz_state {
    uint64_t edges[2];
    int16_t btc2[2];     /* 2 * boxes_to_close[p] (the reference stores x.5 floats) */
    uint8_t to_play;
    int8_t just_played;  /* -1 == None */
    uint8_t flags;       /* engine-internal inside a tree node; 0 in user buffers */
    uint8_t depth;       /* engine-internal */
    int32_t parent;      /* engine-internal */
    int16_t parent_action;
    int16_t result;      /* engine-internal cache of get_result(), DBAZ_RESULT_NONE if None */
} dbaz_state;

typedef struct dbaz_config {
    int32_t abi_version;   /* DBAZ_ABI_VERSION */
    int32_t device;        /* CUDA device ordinal */
    int32_t board_l, board_c; /* BoxesState.BOARD_DIM (dots_boxes_game.py:23) */
    int32_t n_games;       /* concurrent games == trees on this GPU */
    int32_t max_nodes;     /* node-pool capacity per tree (>= sims per move + retained subtree) */
    int32_t lut_size;      /* entries of the host-libm log table for the PUCT constant; 0 = max(65536, 128 * (max_nodes + 1)): every reachable visit count */
    int32_t max_pending;   /* largest max_pending_evals (in-flight simulations per tree) a search may ask for; 0 = 1 */
    double cpuct;          /* UCTNode.CPUCT (mcts.py:44) */
    double cpuct_base;     /* UCTNode.CPUCT_BASE (mcts.py:45) */
} dbaz_config;

typedef struct dbaz_engine dbaz_engine;

/* element type codes for board-plane tensors */
enum { DBAZ_F32 = 0, DBAZ_F16 = 1, DBAZ_BF16 = 2, DBAZ_I16 = 3 };
/* plane layouts */
enum { DBAZ_NCHW = 0, DBAZ_NHWC = 1 };

int dbaz_abi_version(void);
int dbaz_sizeof_state(void);

/* Lifecycle.  Allocates the node pool (n_games * max_nodes * (32 + 16*A) bytes)
 * and per-tree tables on `device`. */
int dbaz_engine_create(const dbaz_config *cfg, dbaz_engine **out);
void dbaz_engine_destroy(dbaz_engine *e);
const char *dbaz_last_error(const dbaz_engine *e); /* e may be NULL: error of the last failed create */
int dbaz_engine_info(const dbaz_engine *e, int32_t *out8); /* {L, C, A, F=3*(L+1)*(C+1), n_games, max_nodes, node_bytes, max_pending} */
/* mcts.py:205 -- UCT_search assigns UCTNode.CPUCT/CPUCT_BASE on every call (host sync: rebuilds the log table) */
int dbaz_engine_set_cpuct(dbaz_engine *e, double cpuct, double cpuct_base);

/* ---- batched game rules over packed states (device arrays of n states) ---- */
/* BoxesState.__init__ (dots_boxes_game.py:30-39) */
int dbaz_game_init(dbaz_engine *e, dbaz_state *states, int64_t n, uint64_t stream);
/* get_valid_moves (dots_boxes_game.py:44-49): out uint8[n][A], 1 = legal */
int dbaz_game_valid_moves(dbaz_engine *e, const dbaz_state *states, uint8_t *out, int64_t n, uint64_t stream);
/* play_ (dots_boxes_game.py:61-89): n_closed int32[n] = number of boxes closed, or -1 where the
 * reference raises ValueError (state left untouched); closed_lc int32[n][4] (may be NULL) = the
 * (l, c) pairs in the reference's order, -1 padded. */
int dbaz_game_play(dbaz_engine *e, dbaz_state *states, const int32_t *moves, int32_t *n_closed,
                   int32_t *closed_lc, int64_t n, uint64_t stream);
/* get_result (dots_boxes_game.py:51-59): int8[n], DBAZ_RESULT_NONE for None */
int dbaz_game_result(dbaz_engine *e, const dbaz_state *states, int8_t *out, int64_t n, uint64_t stream);
/* get_features + nn_batch_builder (dots_boxes_game.py:96-100,148-155): planes[n][3][L+1][C+1]
 * (or NHWC) written directly in the net's input dtype */
int dbaz_game_features(dbaz_engine *e, const dbaz_state *states, void *planes, int32_t dtype, int32_t layout,
                       int64_t n, uint64_t stream);
/* Uniform random legal playouts to terminal (BASELINE config 3).  Move of game g at ply p is the
 * floor(Philox4x32-10(key=seed, ctr=(game0+g, p)) * k / 2^32)-th legal action.  n_plies int32[n];
 * moves uint8[n][max_plies] (may be NULL). */
int dbaz_game_random_rollout(dbaz_engine *e, dbaz_state *states, uint64_t seed, uint64_t game0, int32_t *n_plies,
                             uint8_t *moves, int32_t max_plies, int64_t n, uint64_t stream);

/* ---- search: one tree per game, strictly sequential simulations per tree ---- */
/* create_root_uct_node (mcts.py:156-160) for all n_games trees */
int dbaz_search_reset_roots(dbaz_engine *e, const dbaz_state *root_states, uint64_t stream);
/* Head of UCT_search (mcts.py:205-229).  num_reads int32[n_games] (-1 = tree idle this search;
 * -2 = only the initial _search() of an unexpanded root, without the prior mix; -3 = leave the tree alone: it is in
 * the middle of a search started by an earlier call -- trees need not start their searches together).
 * pending = max_pending_evals (1 <= pending <= cfg.max_pending): simulations in flight per tree.  With 1 the
 * simulations of a tree are strictly sequential; with K the engine reproduces the waves the reference's event loop
 * runs when the net suspends each _search() once (mcts.py:228-242): K select_leaf()s back to back, each leaving its
 * virtual loss behind, a terminal leaf backed up on the spot, then the K expand/backup pairs in the same order; the
 * first wave of a search is min(K, A) wide.
 * noise float64[n_games][A] = Dirichlet sample already multiplied by the legal mask (mcts.py:220-223) or NULL when
 * alpha <= 0; coeff = dirichlet[1].  Unexpanded roots get the extra initial _search() (mcts.py:207-208) before the
 * prior mix, exactly as the reference orders it.  The noise buffer must stay valid until the search has finished. */
int dbaz_search_begin(dbaz_engine *e, const int32_t *num_reads, int32_t pending, const double *noise, double coeff,
                      uint64_t stream);
/* One lock-step wave = for every tree: [expand + backup of its pending leaves, in selection order, using
 * priors/values] then [up to `pending` x (select_leaf + lazy child creation + feature gather)]
 * (mcts.py:105-132,184-199).  All per-leaf buffers have pending * n_games rows; the row of in-flight slot k of
 * tree t is k * n_games + t (so with pending == 1 row == tree).
 *   priors float32[rows][A], values float32[rows]: net outputs for the leaves emitted by the PREVIOUS step
 *   (probabilities, i.e. exp(log_softmax), and tanh value; nn.py:155-160).
 *   planes: net input for the leaves selected by THIS step; leaf_states (may be NULL): their packed states;
 *   leaf_kind int8[rows] (may be NULL): 1 = row holds a leaf that needs evaluation, 0 = empty row.  Terminal leaves
 *   never appear: their simulation is completed inside the step, as in the reference where it never awaits. */
int dbaz_search_step(dbaz_engine *e, const float *priors, const float *values, void *planes, int32_t dtype,
                     int32_t layout, dbaz_state *leaf_states, int8_t *leaf_kind, uint64_t stream);
/* UCT_search's wall-clock limit (mcts.py:201-203,232-233): no tree starts another simulation; the
 * next dbaz_search_step() only backs up the leaves already pending. */
int dbaz_search_stop(dbaz_engine *e, uint64_t stream);
/* root.child_number_visits (mcts.py:244): int32[n_games][A] */
int dbaz_search_root_visits(dbaz_engine *e, int32_t *out, uint64_t stream);
/* Root node view: any of W float32[n][A], priors float64[n][A], sign int32[n][A], ucb float64[n][A]
 * (children_ucb_score, mcts.py:91-99) may be NULL. */
int dbaz_search_root_children(dbaz_engine *e, float *W, double *priors, int32_t *sign, double *ucb, uint64_t stream);
/* Per tree int32[8]: {root_N, max_deepness, tree_size, terminal_count, is_expanded, is_terminal,
 * n_nodes, error}; root_W float32[n]; q float32[n] (TreeRoot.get_tree_stats, mcts.py:33-36) */
int dbaz_search_tree_stats(dbaz_engine *e, int32_t *stats8, float *root_W, float *q, uint64_t stream);
int dbaz_search_root_states(dbaz_engine *e, dbaz_state *out, uint64_t stream);
/* Any node of a tree, for walks from the host (UCTNode.children[...], print_mcts_tree; mcts.py:47-65,247-272).  Node 0 is
 * the root; child[a] (int32[A]) is the node index of the child created for action a, 0 = not created.  W float32[A],
 * N int32[A], priors float64[A], sign int32[A], ucb float64[A] as children_ucb_score() returns them for this node;
 * own8 int32[8] = {own N, is_expanded, is_terminal, parent node, parent action, depth, nodes in the tree, 1 if no such node};
 * own_W float32[1]; state_out: the node's packed state.  Indices are valid until the next dbaz_search_advance_roots /
 * dbaz_search_reset_roots of that tree (re-rooting compacts the pool). */
int dbaz_search_node(dbaz_engine *e, int32_t tree, int32_t node, dbaz_state *state_out, float *W, int32_t *N,
                     double *priors, int32_t *child, int32_t *sign, double *ucb, int32_t *own8, float *own_W,
                     uint64_t stream);
/* int8[n_games]: 1 while the tree's search is running (simulations left or a leaf waiting for the evaluator) */
int dbaz_search_tree_busy(dbaz_engine *e, int8_t *out, uint64_t stream);
/* init_mcts_tree (mcts.py:163-180): moves int32[n_games], -1 = leave that tree alone.  With
 * reuse != 0 the chosen child's subtree is kept (compacted in place), else a fresh root. */
int dbaz_search_advance_roots(dbaz_engine *e, const int32_t *moves, int32_t reuse, uint64_t stream);
/* ---- between two searches of one game, on the device (the asynchronous self-play loop) ----
 * SelfPlay.get_next_move (self_play.py:27-49) and the body of SelfPlay.play_game (self_play.py:51-74) for every tree whose
 * search has finished, while the others keep searching.  All pointers are device memory of the caller; n = n_games,
 * A = the engine's action count.  The per-move tables have n_moves rows (move index = number of moves the game has made). */
typedef struct dbaz_selfplay_buffers {
    int32_t n_moves;
    int32_t reserved;
    const double *inv_temp;    /* [n_moves] 1 / temperature at move index m (self_play.py:29-33) */
    const double *uniforms;    /* [n_moves][n] the uniform of np.random.choice (self_play.py:35) for (move index, tree) */
    const double *noise;       /* [n_moves][n][A] Dirichlet samples over all A entries (mcts.py:220-222); NULL: no noise */
    const int32_t *reads_by_k; /* [A + 1] simulations of a search from a position with k legal moves (self_play.py:41-44) */
    int8_t *searching;         /* [n] in/out: 1 while the tree's game goes on */
    int64_t *move_idx;         /* [n] in/out: move index of the tree's current search */
    int32_t *moves;            /* [n] out: the drawn move of a tree whose search has finished, else -1 (dbaz_search_advance_roots' input) */
    dbaz_state *h_states;      /* [n_moves][n] history of searched roots: packed state ... */
    int32_t *h_visits;         /* [n_moves][n][A] ... root.child_number_visits ... */
    int8_t *h_active;          /* [n_moves][n] ... 1 where a row was recorded ... */
    int32_t *h_moves;          /* [n_moves][n] ... the move played from it ... */
    int32_t *h_stats;          /* [n_moves][n][8] ... dbaz_search_tree_stats' int32[8] ... */
    float *h_q;                /* [n_moves][n] ... and q */
    double *noise_buf;         /* [n][A] the noise array dbaz_search_begin reads: rows of restarting trees are rewritten */
    int32_t *reads;            /* [n] out: dbaz_search_begin's num_reads (-3 = leave the tree alone) */
    int32_t *left;             /* [1] out: games still going on after dbaz_selfplay_restart */
} dbaz_selfplay_buffers;
/* Trees with searching != 0 and no search in progress: the searched root goes into history row move_idx, the move is the
 * first action whose running sum of (visits / max visits)^(1/T) exceeds uniform * total (np.random.choice's searchsorted
 * on the cdf); moves[t] = -1 for every other tree. */
int dbaz_selfplay_pick(dbaz_engine *e, const dbaz_selfplay_buffers *bufs, uint64_t stream);
/* After dbaz_search_advance_roots(moves): trees with moves[t] >= 0 (all trees if first != 0, the start of a batch of
 * games; move_idx is then not advanced) whose game goes on get reads = reads_by_k[legal moves] and their noise row times the
 * legal mask (mcts.py:223); the others get reads = -3.  Follow with dbaz_search_begin(reads, noise_buf, ...). */
int dbaz_selfplay_restart(dbaz_engine *e, const dbaz_selfplay_buffers *bufs, int32_t first, uint64_t stream);
/* Optional, after dbaz_selfplay_restart and before dbaz_search_begin (same `first`): adjudication with the exact endgame
 * solver below.  A tree that restarted (moves[t] >= 0, or first != 0) with searching[t] == 1 and whose root has at most
 * max_free (0 .. 16) free real edges ends its game there: margin[t] = the root's final margin (int8, seen by its player
 * to move), searching[t] = 0, reads[t] = -3 and *left is decremented, so that *left still counts the games going on.
 * margin[t] of every other tree is not written (initialise it to -128).  Capturable in a CUDA graph. */
int dbaz_selfplay_adjudicate(dbaz_engine *e, const dbaz_selfplay_buffers *bufs, int8_t *margin, int32_t max_free,
                             int32_t first, uint64_t stream);
/* Optional instead of dbaz_selfplay_adjudicate, at the same place and with the same trees: exact play.  A tree that
 * restarted with searching[t] == 1 and whose root has at most max_free (0 .. 16) free real edges is played out from there
 * to the first state with a result, with optimal moves (kind 0: outcome-optimal, 1: margin-optimal) and no search.  Ply j
 * writes history row move_idx[t] + j as dbaz_selfplay_pick writes a searched root: h_states = the state, h_visits = 1 on the
 * optimal moves and 0 elsewhere, h_stats and h_q = 0, h_moves = the move drawn from uniforms[move_idx[t] + j][t] with the
 * weights 1, h_active = 1.  Then exact_margin[t] = the root's final margin (int8, seen by its player to move),
 * move_idx[t] = the last row written, searching[t] = 0, reads[t] = -3 and *left is decremented.  The tree's nodes are not
 * touched (its root stays the exact root); exact_margin[t] of every other tree is not written (initialise it to -128).
 * Capturable in a CUDA graph. */
int dbaz_selfplay_exact_endgame(dbaz_engine *e, const dbaz_selfplay_buffers *bufs, int8_t *exact_margin, int32_t max_free,
                                int32_t kind, int32_t first, uint64_t stream);
/* Synchronises `stream`.  out int64[8] = {trees with an error flag, total sims, total path nodes,
 * largest node-pool use of any tree (now or at a re-root), terminal leaves, eval-cache hits, 0, 0} (since reset_roots).  Returns non-zero (and sets
 * last_error) if any tree faulted. */
int dbaz_search_status(dbaz_engine *e, int64_t *out8, uint64_t stream);

/* ---- lock-step scheduling extras (max_pending_evals == 1 searches) ----
 * compact != 0: the leaf a tree hands to the evaluator goes to the next free row of the batch (rows 0..n-1 are the
 * n leaves of the wave, in no particular order) instead of row == tree, so the evaluator only has to run as many rows
 * as there are busy trees; leaf_kind is not written in this mode.  max_inline > 0 bounds how many simulations of one
 * tree may complete inside one dbaz_search_step() without the evaluator (terminal leaves, eval-cache hits); 0 = no
 * bound: a tree runs on until a leaf needs the net (the order of a tree's simulations, hence every result, is the
 * same for any setting). */
int dbaz_search_set_mode(dbaz_engine *e, int32_t compact, int32_t max_inline);
/* A second bound on the in-kernel chains of dbaz_search_set_mode: a tree starts no further net-free simulation once it has
 * spent `microseconds` in a dbaz_search_step launch (0 = no time bound, the default).  A launch lasts as long as its longest
 * chain; the time bound lets trees whose simulations are cheap run on while the launch waits for the expensive ones.  Like the
 * count, it only shapes the schedule: results are the same for every value.  Captured launches keep the value they were
 * captured with. */
int dbaz_search_set_chain_budget(dbaz_engine *e, int32_t microseconds);
/* Compact mode: the evaluator that follows the next dbaz_search_step() calls will run rows 0..rows-1 only
 * (0 = no limit).  A tree whose leaf would land beyond them drops that selection and repeats it in the next wave --
 * the selection wrote nothing but a lazily created child, so the repeat finds the same leaf over the same path and
 * no result changes; it only costs the repeat.  Lets the host size the evaluator's batch by the rows recent waves
 * actually asked for instead of by the number of busy trees. */
int dbaz_search_set_batch_rows(dbaz_engine *e, int32_t rows);
/* Enqueues a copy of {rows the most recent dbaz_search_step() asked for, trees that still have work after it
 * (after dbaz_search_begin(): trees with simulations to run), largest rows figure since the previous call, 0} on
 * `stream` into out4 (int32[4], device or pinned host memory).  The busy-tree count never grows during a search, so
 * a stale value is a safe upper bound of the next wave's rows. */
int dbaz_search_wave_counts(dbaz_engine *e, int32_t *out4, uint64_t stream);

/* ---- one CUDA graph per search: the adaptive wave loop without the host (dotsboxesaz_b200/csrc/dbaz_loop.cuh) ----
 * rung_graphs[r]: a cudaGraph_t (not instantiated; e.g. torch.cuda.CUDAGraph(keep_graph=True).raw_cuda_graph()) holding
 * some waves of [dbaz_search_step -> evaluator] captured with dbaz_search_set_batch_rows(rung_rows[r]); rung_rows strictly
 * descending; rung_us[r] the measured evaluator time of that batch.  The built graph is: a begin kernel (first rung from
 * the busy-tree count dbaz_search_begin left), a WHILE conditional node (trees still busy) around a SWITCH conditional
 * node over the rung graphs (cloned as child graphs) and a decision kernel that reads the wave counters and picks the
 * next rung (most rows served per microsecond; a rung up to `undersize` short when `undersize_gain` cheaper per row).
 * max_iters bounds the replays of one launch.  Call dbaz_search_begin, then dbaz_search_loop_launch: when the launch has
 * drained, every tree has finished its search.  dbaz_search_loop_counts copies the per-rung replay counts since the last
 * call to replays_out (uint32[n_rungs], device or pinned host) and zeroes them, in stream order. */
int dbaz_search_loop_build(dbaz_engine *e, const uint64_t *rung_graphs, const int32_t *rung_rows, const float *rung_us,
                           int32_t n_rungs, int32_t max_iters, float row_margin, float undersize, float undersize_gain,
                           float wave_overhead_us, uint64_t *loop_out);
/* The decision rule of the loop's device kernel, callable on the host (no GPU needed): index of the rung chosen for
 * waves expected to ask for `want` rows. */
int dbaz_search_loop_pick(const int32_t *rung_rows, const float *rung_us, int32_t n_rungs, float undersize,
                          float undersize_gain, float wave_overhead_us, int32_t want);
int dbaz_search_loop_launch(dbaz_engine *e, uint64_t loop, uint64_t stream);
int dbaz_search_loop_counts(dbaz_engine *e, uint64_t loop, uint32_t *replays_out, uint64_t stream);
void dbaz_search_loop_destroy(dbaz_engine *e, uint64_t loop);

/* ---- evaluation cache: the engine's form of AsyncBatchedProxy's LRU (utils/proxies.py:23-26,35-43) ----
 * A direct-mapped device table of 2^log2_entries entries (16*A bytes each) keyed by get_hash() = (edge set,
 * boxes_to_close[to_play]) (dots_boxes_game.py:106-112), shared by all trees of the engine.  The step kernel
 * stores every (priors, value) the evaluator returns and, for max_pending_evals == 1 searches, completes a
 * simulation whose leaf is found in the table on the spot -- as the reference's proxy returns a cached result
 * without suspending.  Keys are compared exactly (all 136 bits: 128 edge bits + the counter), so a hit always returns an
 * evaluation of the same features.  log2_entries == 0 frees the table.  Synchronises the device. */
int dbaz_cache_configure(dbaz_engine *e, int32_t log2_entries);
/* Forget every entry (call after the net's weights change).  O(1): the keys carry a table epoch, which this call bumps. */
int dbaz_cache_clear(dbaz_engine *e, uint64_t stream);

/* ---- leaf-evaluation pipeline: fused stages around the library GEMMs/convs ----
 * (replace the separate gather / bias / ReLU / eval-BatchNorm / softmax passes of NeuralNetWrapper.predict_sync,
 * nn.py:155-160, around dots_boxes_nn.py:85-98 and nn.py:49-58).  scale/shift are the folded eval-mode BatchNorm
 * (gamma/sqrt(var+eps), beta - mean*scale), float32[channels]. */
/* Leaf gather + first 3x3 conv (zero padding 1, 3 input planes) + epilogue in one kernel, reading the packed
 * leaf states instead of a plane tensor (dots_boxes_game.py:96-100 + dots_boxes_nn.py:85 / nn.py:118-119,27-28).
 * w01 float32[2][3][3][cout]: weights of the two edge planes; bias_pos / k2_pos float32[(L+1)*(C+1)][cout]:
 * position-dependent constant and coefficient of the third plane's value (host-folded: conv bias, in-board
 * taps of plane 2, optional input BatchNorm).  out [n][L+1][C+1][cout] (NHWC) bf16/fp16.
 * mode 0: scale*relu(y)+shift, mode 1: relu(scale*y+shift). */
int dbaz_nn_stem(dbaz_engine *e, const dbaz_state *leaf_states, const float *w01, const float *bias_pos, const float *k2_pos,
                 const float *scale, const float *shift, void *out, int32_t cout, int32_t dtype, int32_t mode, int64_t n,
                 uint64_t stream);
/* The same stem as one tensor-core implicit GEMM (K = 48, fp32 accumulate, ReLU).  Weights: w48 [48][cout] in the
 * output dtype (16-bit), rows 0-17 the two edge planes' taps (plane, ky, kx), 18-26 the third plane's taps, 27-35
 * per-tap constants that apply where the tap lies inside the board (input BatchNorm shift), 36 the bias, 37-47 zero;
 * any output affine is folded into w48 by the caller.  dbaz_nn_stem_mma_pack() reorders them once into the
 * tensor-core fragment order (`packed`: 48*cout elements), which dbaz_nn_stem_mma() takes.
 * out [n][L+1][C+1][cout] (NHWC) bf16/fp16; cout a multiple of 64. */
int dbaz_nn_stem_mma_pack(dbaz_engine *e, const void *w48, void *packed, int32_t cout, uint64_t stream);
int dbaz_nn_stem_mma(dbaz_engine *e, const dbaz_state *leaf_states, const void *packed, void *out, int32_t cout, int32_t dtype,
                     int64_t n, uint64_t stream);
/* logits [n][ld], ld >= A + 1: columns 0..A-1 policy logits, column A value pre-activation ->
 * priors float32[n][A] = softmax (exp(log_softmax)), values float32[n] = tanh. */
int dbaz_nn_heads(dbaz_engine *e, const void *logits, int32_t ld, int32_t dtype, float *priors, float *values, int64_t n,
                  uint64_t stream);

/* dbaz_nn_heads with ResNetZero's value head finished in the kernel (ValueHead.forward, nn.py:95-97): columns A .. A + n_hidden - 1
 * of a row are the hidden layer's pre-activations; values = tanh(v_w[n_hidden] + sum_j relu(h_j) * v_w[j])
 * (v_w float32[n_hidden + 1] on the device: fc1's weights, then its bias). */
int dbaz_nn_heads_mlp(dbaz_engine *e, const void *logits, int32_t ld, int32_t dtype, int32_t n_hidden, const float *v_w,
                      float *priors, float *values, int64_t n, uint64_t stream);

/* ---- residual tower of ResNetZero as ONE persistent tcgen05 kernel (dotsboxesaz_b200/csrc/dbaz_tower.cu) ----
 * Replaces the 2 * nb_blocks conv3x3 -> BatchNorm -> ReLU (-> +x) library calls of ResNet.forward / ResBlock.forward
 * (nn.py:16-30,33-58; 20 blocks of 64 channels in configuration.py:133-155) and, optionally, the two 1x1 head
 * convolutions + BatchNorm + ReLU (PolicyHead / ValueHead conv0, nn.py:80,95).  64 channels, boards with L + 1 <= 6.
 *
 * dbaz_nn_tower_geometry: out8 = {supported, boards per tile, plane bytes, tile bytes, weight chunk bytes (6144),
 *   chunks per stage (12), channels (64), padded row width C + 2}.
 * Activations enter as "planar tiles" (tile t = boards [t * nb, (t + 1) * nb)): tile_bytes per tile, byte
 *   128 + cg * plane + ((h * 128) + b * (C + 2) + w) * 16 + 2 * (c % 8)  holds channel c = 8 cg + c % 8 of point (h, w) of
 *   board b of the tile; every other byte must be zero (allocate zero-filled once; dbaz_nn_tower_planarize writes only
 *   real points).  dbaz_nn_tower_planarize converts [n][L+1][C+1][64] bf16 (NHWC).
 * packed_w: for stage s (conv1 / conv2 of block s / 2, BatchNorm folded into weight and bias) 12 chunks
 *   p = 4 * kx + ks of 6144 bytes [kh 2][row = 64 * (2 - ky) + cout][8] bf16 = weight[cout][16 ks + 8 kh + i][ky][kx];
 *   then, if head_cout, one chunk [ks 4][kh 2][cout][8] of the 1x1 head weights.  bias float32[n_stages (+1)][64].
 * out: [n][L+1][C+1][head_cout ? head_cout : 64] bf16 = relu(head(tower(x))) resp. tower(x).
 * Stage s odd adds the input of stage s - 1 (the residual) before the ReLU.  head_cout in {0, 16, 32}. */
int dbaz_nn_tower_geometry(dbaz_engine *e, int32_t *out8);
/* dbaz_nn_stem_mma() (64 output channels, bf16) writing planar tiles directly: stem -> tower without an NHWC pass. */
int dbaz_nn_stem_mma_tiles(dbaz_engine *e, const dbaz_state *leaf_states, const void *w48, void *tiles, int64_t n,
                           uint64_t stream);
int dbaz_nn_tower_planarize(dbaz_engine *e, const void *nhwc, void *tiles, int64_t n, uint64_t stream);
int dbaz_nn_tower(dbaz_engine *e, const void *tiles, const void *packed_w, const float *bias, int32_t n_stages,
                  int32_t head_cout, void *out, int64_t n, uint64_t stream);
/* Diagnostics: later dbaz_nn_tower() launches record a clock64 timeline of CTA 0's first tile into timeline
 * (device int64[64][16]: per stage {MMA: stage start, weights of pass 0 / 1 landed, last MMA issued; epilogue of
 * h-block h: accumulator ready, block written}); NULL switches it off. */
int dbaz_nn_tower_trace(dbaz_engine *e, int64_t *timeline);

/* ---- one 256-channel 3x3 convolution of SimpleNN's trunk as a tcgen05 GEMM per output position
 *      (dotsboxesaz_b200/csrc/dbaz_trunk.cu) ----
 * y[b][p][:] = relu((sum over the taps t of p inside the grid: x[b][q_t][:] . w[t] + bias_pos[p][:]) + bias[:]), bf16 in
 * and out, fp32 accumulation and epilogue; the taps that fall into the zero padding are never loaded or multiplied.  Each
 * output element is accumulated in one fixed order (64-channel chunks ascending, in-board taps by (ky, kx) inside a
 * chunk), so a board's output does not depend on n or on the row it sits in; it is cuDNN's order for the same conv, so
 * with bf16-valued biases the result equals cuDNN's conv-add-bias-ReLU with z = bias_pos.
 *
 * dbaz_nn_trunk_conv_taps (no engine, no device): the tap table of a 3x3 convolution with zero padding pad (0 or 1) over
 *   an hi x wi grid (hi * wi <= 64).  out: int32[2 + 10 * 64 + 64] = {ho, wo; for output position p = y * wo + x < ho * wo:
 *   the tap count, then (q << 8) | (3 ky + kx) for each in-board tap by ascending (ky, kx), -1 beyond; then the output
 *   positions in the order the kernel hands them out (descending tap count), -1 beyond}.  Returns 1 on a bad shape.
 * dbaz_nn_trunk_conv_plan: binds one layer's buffers once and writes dbaz_nn_trunk_conv_plan_bytes() bytes to the host
 *   buffer plan -- the tensor maps over the full capacity, so dbaz_nn_trunk_conv encodes and allocates nothing (safe
 *   inside a stream capture).  x: [cap][hi][wi][256] bf16 (NHWC); y: [cap][ho][wo][256] bf16; packed_w: [ky][kx][cout][cin]
 *   bf16; bias_pos: [ho * wo][256] float32; bias: [256] float32.  All 16-byte aligned; the buffers must outlive the plan.
 * dbaz_nn_trunk_conv: runs the layer for boards 0 .. n-1 (n <= cap); rows n .. cap-1 of y are not written. */
int dbaz_nn_trunk_conv_taps(int32_t hi, int32_t wi, int32_t pad, int32_t *out);
int64_t dbaz_nn_trunk_conv_plan_bytes(void);
int dbaz_nn_trunk_conv_plan(dbaz_engine *e, const void *x, void *y, const void *packed_w, const float *bias_pos, const float *bias, int64_t cap,
                            int32_t hi, int32_t wi, int32_t pad, void *plan);
int dbaz_nn_trunk_conv(dbaz_engine *e, const void *plan, int64_t n, uint64_t stream);

/* ---- test/bench utility: deterministic stand-in for the policy/value net ----
 * (SURVEY.md 8a KAT definition; kind 0 hash-seeded, kind 1 uniform prior) over leaf_states[n]. */
int dbaz_fake_nn(dbaz_engine *e, const dbaz_state *leaf_states, float *priors, float *values, int32_t kind,
                 int64_t n, uint64_t stream);

/* ---- exact solver for boards of at most 32 real edges (dotsboxesaz_b200/csrc/dbaz_solver.cuh, DESIGN.md §10) ----
 * E = 2LC + L + C real edges; compact edge j = the j-th real action in increasing order; M = played edges as a 32-bit
 * compact mask.  table: caller-owned int8[2^E], entry M = v(M), the largest net number of boxes the player to move can
 * still gain against best play (full-game recurrence, no early stop).  The mover's lead d = LC - btc2[to_play] - closed
 * boxes; final margin = d + v(M), outcome = sign(final margin), both seen by the player to move.  Every entry point rejects
 * boards with E > 32 (4x4 and up) with an error message.
 * dbaz_solver_solve: fills the table (one kernel per popcount layer) and checks that every entry was written;
 * table_bytes must be 2^E.  Synchronises `stream`. */
int dbaz_solver_solve(dbaz_engine *e, int8_t *table, int64_t table_bytes, uint64_t stream);
/* move_margin int8[n][A]: d + (c > 0 ? c + v(M|a) : -v(M|a)) for every free edge a (c = boxes a closes), -128 for
 * played edges and padding; margin int8[n]: the final margin. */
int dbaz_solver_moves(dbaz_engine *e, const int8_t *table, const dbaz_state *states, int8_t *move_margin, int8_t *margin,
                      int64_t n, uint64_t stream);
/* A perfect-play evaluator for dbaz_search_step's leaves: priors float32[n][A] = 1/k (k = __fdiv_rn(1, k)) on the k moves
 * whose margin has the sign of the outcome, 0 elsewhere; values float32[n] = outcome (mode 0) or final margin / (L C)
 * (mode 1).  A function of the eval-cache key; no allocation and no synchronisation (capturable in a CUDA graph). */
int dbaz_solver_eval(dbaz_engine *e, const int8_t *table, const dbaz_state *leaf_states, float *priors, float *values,
                     int32_t mode, int64_t n, uint64_t stream);

/* ---- exact endgame solver for every board (dotsboxesaz_b200/csrc/dbaz_endgame.cuh, DESIGN.md §11) ----
 * A state with f free real edges is solvable when f <= max_free; max_free must be in [0, 16].  Its value v(M) (as above)
 * comes from a retrograde over the 2^f subsets of its free edges, in shared memory, so no table is needed and every
 * board the engine plays is supported.  Margins, outcomes and move margins are those of the solver entries above.
 * Neither entry allocates or synchronises (both are capturable in a CUDA graph).
 * dbaz_endgame_moves: move_margin int8[n][A] and margin int8[n] as dbaz_solver_moves for solvable states; every byte of
 * an unsolvable state's row and its margin is -128. */
int dbaz_endgame_moves(dbaz_engine *e, const dbaz_state *states, int8_t *move_margin, int8_t *margin, int32_t max_free,
                       int64_t n, uint64_t stream);
/* An endgame-exact evaluator, run after another evaluator on the same leaves: it rewrites only the rows of solvable
 * leaves, with priors as dbaz_solver_eval (left as they are when keep_priors != 0) and values = outcome (mode 0) or final
 * margin / (L C) (mode 1).  Every other row keeps its bits.  A function of the eval-cache key. */
int dbaz_endgame_eval(dbaz_engine *e, const dbaz_state *leaf_states, float *priors, float *values, int32_t mode,
                      int32_t keep_priors, int32_t max_free, int64_t n, uint64_t stream);
/* Deep tier (DESIGN.md §13): every one of the n states has exactly f free real edges, 17 <= f <= 32.  Each is solved in a
 * 2^f-byte table of its own in the caller-owned device workspace, by the layer kernel of dbaz_solver_solve over its free
 * edges; a position takes 2^f + 512 bytes of workspace (table and geometry), and the states are solved in passes of as
 * many positions as the workspace holds (at most 65 535).  Outputs as dbaz_endgame_moves: move_margin int8[n][A] (-128
 * for played edges and padding) and margin int8[n].  Rejects f outside [17, 32], a workspace smaller than one position,
 * null buffers, n < 0, states whose f differs and unwritten table entries.  Allocates an 8-byte counter and synchronises
 * `stream`; not capturable. */
int dbaz_endgame_deep_moves(dbaz_engine *e, const dbaz_state *states, int64_t n, int32_t f, int8_t *workspace,
                            int64_t workspace_bytes, int8_t *move_margin, int8_t *margin, uint64_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DBAZ_B200_H */
