// The per-check phase of the asynchronous self-play loop (BatchedSelfPlay.play_games_async): what the reference does
// between two searches of one game -- SelfPlay.get_next_move (self_play.py:27-49: temperature, draw of the move) and the
// body of SelfPlay.play_game (self_play.py:51-74: record the searched root, re-root, next search) -- for every tree whose
// search has finished, while the other trees keep searching.  Two kernels around the engine's own k_advance_roots:
//
//   k_selfplay_pick     one warp per tree, lane = action: visits -> (v / max)^(1/T) -> running sum -> the first action whose
//                       cumulative weight exceeds u * total (np.random.choice's searchsorted on the cdf, with the uniform
//                       pre-drawn per (move index, tree)); the searched root (state, visits, tree statistics, q) goes
//                       into the history row of its move index; moves[t] = the move, or -1 for trees that are not done.
//   k_selfplay_restart  after the re-root: games that go on get the simulation budget of their number of legal moves
//                       (n_searches) and their row of Dirichlet noise times the legal mask (mcts.py:220-223); the others
//                       are told to leave their tree alone (num_reads = -3, k_search_begin); counts the games still on.
//   k_selfplay_adjudicate  optional, after the restart: a game whose new root has f <= max_free free edges ends there
//                       with the exact final margin of that root (the endgame solver of dbaz_endgame.cuh); its root is
//                       not searched and gives no sample.
//   k_selfplay_exact_endgame  optional instead, at the same place: a game whose new root has f <= max_free free edges is
//                       played out from there with optimal moves by the warp that solves the root, one sample row per
//                       ply with the optimal moves as its visits, and ends with that root's exact final margin.
#pragma once
#include "dbaz_tree_kernels.cuh"
#include "dbaz_endgame.cuh"

namespace dbaz {

struct SelfplayArgs {
    int n_moves;
    const double* inv_temp;    // [n_moves]
    const double* uniforms;    // [n_moves][n]
    const double* noise;       // [n_moves][n][A] or null
    const int32_t* reads_by_k; // [A + 1]
    int8_t* searching;         // [n]
    int64_t* move_idx;         // [n]
    int32_t* moves;            // [n]
    dbaz_state* h_states;      // [n_moves][n]
    int32_t* h_visits;         // [n_moves][n][A]
    int8_t* h_active;          // [n_moves][n]
    int32_t* h_moves;          // [n_moves][n]
    int32_t* h_stats;          // [n_moves][n][8]
    float* h_q;                // [n_moves][n]
    double* noise_buf;         // [n][A]
    int32_t* reads;            // [n]
    int32_t* left;             // [1]
};

constexpr int SP_WARPS = 4;

__global__ void __launch_bounds__(SP_WARPS * 32) k_selfplay_pick(Board b, TreeArgs ta, SelfplayArgs sp) {
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    if (blockIdx.x == 0 && threadIdx.x == 0) *sp.left = 0;  // k_selfplay_restart (a later launch) counts into it
    if (t >= ta.n_trees) return;
    const TreeHot hot = load_hot(ta.trees + t);
    const bool done = sp.searching[t] && !(hot.sims_left > 0 || hot.n_pending > 0);
    if (!done) {
        if (lane == 0) sp.moves[t] = -1;
        return;
    }
    const int A = b.A, n = ta.n_trees;
    const int mi = (int)min((long long)sp.move_idx[t], (long long)sp.n_moves - 1);
    char* np = node_ptr(ta, t, 0);
    const dbaz_state h = load_hdr(np);
    const bool interior = (h.flags & NF_EXPANDED) && !(h.flags & NF_TERMINAL);
    const Child* ch = node_children(np);
    const int64_t row = (int64_t)mi * n + t;
    // ---- visits, their maximum
    int vis[DBAZ_MAX_ACTIONS / 32];
    int vmax = 0;
#pragma unroll
    for (int i = 0; i < DBAZ_MAX_ACTIONS / 32; ++i) {
        const int a = lane + 32 * i;
        vis[i] = (a < A && interior) ? ch[a].N : 0;
        vmax = max(vmax, vis[i]);
        if (a < A) sp.h_visits[row * A + a] = vis[i];
    }
    vmax = __reduce_max_sync(0xffffffffu, vmax);
    // ---- (v / max)^(1/T), running sum in action order, first action beyond u * total
    const double it = sp.inv_temp[mi];
    const double den = (double)max(vmax, 1);
    double carry = 0.0;
    double cdf[DBAZ_MAX_ACTIONS / 32];
    int last_pos = -1;  // the last action with a positive weight
#pragma unroll
    for (int i = 0; i < DBAZ_MAX_ACTIONS / 32; ++i) {
        const int a = lane + 32 * i;
        double p = vis[i] > 0 ? pow((double)vis[i] / den, it) : 0.0;
        if (a >= A) p = 0.0;
        const unsigned pos = __ballot_sync(0xffffffffu, p > 0.0);
        if (pos) last_pos = 32 * i + 31 - __clz(pos);
        double s = p;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double o = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += o;
        }
        cdf[i] = carry + s;
        carry = __shfl_sync(0xffffffffu, cdf[i], 31);
    }
    const double target = sp.uniforms[row] * carry;
    int move = -1;
#pragma unroll
    for (int i = 0; i < DBAZ_MAX_ACTIONS / 32; ++i) {
        const int a = lane + 32 * i;
        const unsigned beyond = __ballot_sync(0xffffffffu, a < A && cdf[i] > target);
        if (move < 0 && beyond) move = 32 * i + __ffs(beyond) - 1;
    }
    if (move < 0) move = last_pos;  // u * total rounded up to the total
    if (lane == 0) {
        dbaz_state pub = h;
        pub.flags = 0; pub.depth = 0; pub.parent = -1; pub.parent_action = -1; pub.result = (int16_t)state_result(h);
        sp.h_states[row] = pub;
        const TreeRec T = ta.trees[t];
        int32_t* o = sp.h_stats + row * 8;
        o[0] = T.root_N; o[1] = T.max_deepness - T.deepness_correction; o[2] = T.tree_size; o[3] = T.terminal_count;
        o[4] = (h.flags & NF_EXPANDED) ? 1 : 0; o[5] = (h.flags & NF_TERMINAL) ? 1 : 0; o[6] = T.n_nodes;
        o[7] = (int32_t)(T.flags & (TF_ERR_POOL | TF_ERR_MOVE));
        sp.h_q[row] = __fdiv_rn(T.root_W, (float)(1 + T.root_N));  // mcts.py:35
        sp.h_moves[row] = move;
        sp.h_active[row] = 1;
        sp.moves[t] = move;
        if (move < 0) sp.searching[t] = 0;  // a finished search without a single visit (cannot happen for a legal budget): the
                                            // game stops here instead of being picked up again at every check
    }
}

// first != 0: the start of a batch of games -- every tree begins its first search, no move has been drawn
template <int NW>
__global__ void __launch_bounds__(SP_WARPS * 32) k_selfplay_restart(Board b, TreeArgs ta, SelfplayArgs sp, int first) {
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    if (t >= ta.n_trees) return;
    const bool done = first || sp.moves[t] >= 0;
    if (!done) {
        if (lane == 0) {
            sp.reads[t] = -3;
            if (sp.searching[t]) atomicAdd(sp.left, 1);
        }
        return;
    }
    const int A = b.A, n = ta.n_trees;
    const long long next = first ? sp.move_idx[t] : sp.move_idx[t] + 1;
    const dbaz_state h = load_hdr(node_ptr(ta, t, 0));  // the new root
    const bool go_on = state_result(h) == DBAZ_RESULT_NONE && next < sp.n_moves;
    int k = 0;
    for (int a0 = 0; a0 < A; a0 += 32) {
        const int a = a0 + lane;
        const bool legal = a < A && state_legal<NW>(b, h, a);
        k += __popc(__ballot_sync(0xffffffffu, legal));
        if (go_on && sp.noise && a < A) {
            const int64_t o = (int64_t)t * A + a;
            sp.noise_buf[o] = legal ? sp.noise[((int64_t)next * n) * A + o] : 0.0;  // mcts.py:223: noise * valid_actions
        }
    }
    if (lane == 0) {
        sp.move_idx[t] = next;
        sp.searching[t] = go_on ? 1 : 0;
        sp.reads[t] = go_on ? sp.reads_by_k[k] : -3;
        if (go_on) atomicAdd(sp.left, 1);
    }
}

// Row source of k_selfplay_adjudicate: row t is the root of tree t (node 0 of its pool).  Only trees that restarted at
// this check (first, or a move was drawn) and go on qualify; any other tree is not read.
struct RootRows {
    TreeArgs ta;
    const int8_t* searching;
    const int32_t* moves;
    int first;
    __device__ __forceinline__ bool qualifies(int64_t t) const { return (first || moves[t] >= 0) && searching[t] == 1; }
    __device__ __forceinline__ dbaz_state state(int64_t t) const { return load_hdr(node_ptr(ta, (int)t, 0)); }
};

// A solvable qualifying root ends its game: its final margin goes to margin[t], the tree stops searching, k_search_begin
// leaves it alone and it no longer counts as a game going on.  Every other tree is left as it is.
struct AdjudicateOut {
    int8_t* margin;
    int8_t* searching;
    int32_t* reads;
    int32_t* left;
    static constexpr bool kUnsolvable = false;
    __device__ __forceinline__ void unsolvable(const Board&, int64_t, int) const {}
    __device__ __forceinline__ void solved(const Board&, const EndgameRow& p, const int8_t* T, const uint32_t*, int64_t t,
                                           int lane) const {
        if (lane == 0) {
            margin[t] = (int8_t)(p.d + T[0]);
            searching[t] = 0;
            reads[t] = -3;
            atomicSub(left, 1);
        }
    }
};

__global__ void __launch_bounds__(ENDGAME_THREADS, 3) k_selfplay_adjudicate(Board b, TreeArgs ta, const uint16_t* __restrict__ order,
                                                                        SelfplayArgs sp, int8_t* margin, int max_free, int first) {
    endgame_rows(b, ta.act_tab, order, RootRows{ta, sp.searching, sp.moves, first},
                 AdjudicateOut{margin, sp.searching, sp.reads, sp.left}, max_free, (int64_t)ta.n_trees);
}

// A solvable qualifying root is played out to the end of its game by the warp that solved it, from that one table (DESIGN.md
// §14).  Lane i is local edge i (f <= 16); m = the local edges played since the root, d = the mover's lead (as endgame_lead
// reads it from the state: the boxes closed since the root are counted, the rest comes from btc2).  Per ply, the
// row mi = move_idx[t] + j gets what k_selfplay_pick writes for a searched root: the published state, visits = 1 on the
// optimal moves (kind 0: outcome-optimal, 1: margin-optimal) and 0 elsewhere, zero tree statistics and q, the move drawn
// from uniforms[mi][t] with pick's arithmetic (weights 1.0: a running double sum, the first action beyond u * k, else the
// last positive weight), active = 1.  The game ends at the first state with a result (or a full history).  Then the tree
// ends as in AdjudicateOut, with move_idx[t] = its last row and exact_margin[t] = the root's final margin.  The tree's
// node pool is not touched: its root stays the exact root.
struct ExactOut {
    TreeArgs ta;
    SelfplayArgs sp;
    int8_t* exact_margin;
    int kind;
    static constexpr bool kUnsolvable = false;
    __device__ __forceinline__ void unsolvable(const Board&, int64_t, int) const {}
    __device__ __forceinline__ void solved(const Board& b, const EndgameRow& p, const int8_t* T, const uint32_t* geo, int64_t tw,
                                           int lane) const {
        const int t = (int)tw, n = ta.n_trees, A = b.A;
        const bool mine = lane < p.f;
        const uint32_t bit = 1u << lane;
        const int act = mine ? endgame_action(p.F0, p.F1, __popcll(p.F0), lane) : -1;
        const uint32_t eb = mine ? geo[lane] : 0u, b0 = eb & 0xffffu, b1 = eb >> 16;
        dbaz_state s = load_hdr(node_ptr(ta, t, 0));
        const int64_t mi0 = sp.move_idx[t];
        uint32_t m = 0;
        int closed = b.nboxes - ((s.to_play & 1) ? s.btc2[1] : s.btc2[0]) - p.d;  // boxes closed at the root
        int d = p.d, j = 0;
        for (; state_result(s) == DBAZ_RESULT_NONE && mi0 + j < sp.n_moves; ++j) {
            const int64_t row = (mi0 + j) * n + t;
            const int vm = T[m];
            int c = 0;
            bool opt = false;
            if (mine && !(m & bit)) {
                const uint32_t x = m | bit;
                c = ((b0 && (x & b0) == b0) ? 1 : 0) + ((b1 && (x & b1) == b1) ? 1 : 0);
                const int v = T[x];
                const int mv = c ? c + v : -v;
                opt = kind ? mv == vm : sign_of(d + mv) == sign_of(d + vm);
            }
            const uint32_t om = __ballot_sync(0xffffffffu, opt);
            if (!om) break;  // no free edge left without a result: only a state with inconsistent scores gets here
            for (int a = lane; a < A; a += 32) {
                const bool fr = a < 64 ? ((p.F0 >> a) & 1ull) : ((p.F1 >> (a - 64)) & 1ull);
                sp.h_visits[row * A + a] = fr ? (int32_t)((om >> endgame_rank(p.F0, p.F1, a)) & 1u) : 0;
            }
            // local edges are in action order, so the running count of optimal local edges is pick's cdf
            const double target = sp.uniforms[row] * (double)__popc(om);
            const unsigned beyond = __ballot_sync(0xffffffffu, mine && (double)__popc(om & (bit | (bit - 1u))) > target);
            const unsigned last = __ballot_sync(0xffffffffu, opt && (om >> lane) == 1u);  // the last optimal local edge
            const int i = __ffs(beyond ? beyond : last) - 1;
            const int move = __shfl_sync(0xffffffffu, act, i);
            const int c_i = __shfl_sync(0xffffffffu, c, i);
            if (lane == 0) {
                dbaz_state pub = s;
                pub.flags = 0; pub.depth = 0; pub.parent = -1; pub.parent_action = -1; pub.result = (int16_t)state_result(s);
                sp.h_states[row] = pub;
                int32_t* o = sp.h_stats + row * 8;
#pragma unroll
                for (int k = 0; k < 8; ++k) o[k] = 0;
                sp.h_q[row] = 0.0f;
                sp.h_moves[row] = move;
                sp.h_active[row] = 1;
            }
            state_apply<2>(s, move, c_i);  // two edge words fit every board: the second stays 0 where A <= 64
            closed += c_i;
            d = b.nboxes - ((s.to_play & 1) ? s.btc2[1] : s.btc2[0]) - closed;
            m |= 1u << i;
        }
        if (lane == 0) {
            exact_margin[t] = (int8_t)(p.d + T[0]);
            if (j > 0) sp.move_idx[t] = mi0 + j - 1;  // (no row: a root with a result or a full history, not met in self-play)
            sp.searching[t] = 0;
            sp.reads[t] = -3;
            atomicSub(sp.left, 1);
        }
    }
};

// Two CTAs of 512 threads per SM, not the three of the other endgame kernels: the playout loop does not fit their 40
// registers (it spilled there); it takes 59 here, without spills.
__global__ void __launch_bounds__(ENDGAME_THREADS, 2) k_selfplay_exact_endgame(Board b, TreeArgs ta, const uint16_t* __restrict__ order,
                                                                           SelfplayArgs sp, int8_t* exact_margin, int max_free,
                                                                           int kind, int first) {
    endgame_rows(b, ta.act_tab, order, RootRows{ta, sp.searching, sp.moves, first}, ExactOut{ta, sp, exact_margin, kind}, max_free,
                 (int64_t)ta.n_trees);
}

}  // namespace dbaz
